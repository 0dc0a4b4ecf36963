// Internal types shared by prover.cu (keygen + create_proof) and verifier.cu (verify_proof): the device images of
// Params / VerifyingKey / ProvingKey, the flattened constraint system, the static multiopen structure, and the host transcript.
// Not part of the C ABI (include/bzhalo2.h).
#pragma once
#include "../../include/bzhalo2.h"
#include "common.h"
#include "fixedmsm.h"
#include "poly.cuh"
#include "curve.cuh"
#include "sqrt.cuh"
#include "blake2b.h"
#include <algorithm>
#include <array>
#include <cstdlib>
#include <functional>
#include <map>
#include <set>

typedef bzh::Fe HFe;

namespace bz {

void msm_run_batch(Ctx* ctx, int curve, const void* const* d_main, const void* const* d_extra, uint32_t n_main, uint32_t first, uint32_t n,
                   const void* bases, uint32_t n_msm, void* out_jac);
void msm_multi_run(Ctx* ctx, int curve, const void* scalars, uint32_t nq, const void* bases, uint32_t stride, uint32_t outputs, void* out_jac);
void jac_to_affine_run(Ctx* ctx, int curve, const void* jac, void* aff, uint32_t n);
void jac_sum_run(Ctx* ctx, int curve, const void* d_jac, uint32_t count, void* d_out_affine);
void decompress_points_run(Ctx* ctx, int curve, const void* d_in, void* d_out_affine, uint8_t* d_status, uint32_t count);
void lookup_permute_large_run(Ctx* ctx, const void* cin, const void* ctab, void* aout, void* sout, uint32_t usable, uint32_t* d_err);

typedef ::bz::Fe<FpP> DFe;      // device element type of the prover's scalar field (Vesta scalars = Fp)

// h(X) as generated straight-line code (gen_quotient.cu, emitted by scripts/gen_quotient_kernels.py from the compiled program of a
// known circuit): same arguments as eval_program_kernel, found by the FNV-1a hash of the program words and its rotation table
typedef void (*QuotientLaunchFn)(const EvalArgs<FpP>& a, dim3 grid, cudaStream_t st);
QuotientLaunchFn find_generated_quotient(uint64_t hash);
inline uint64_t program_hash(const std::vector<uint32_t>& code, const std::vector<int32_t>& rot) {
  uint64_t h = 0xcbf29ce484222325ull;
  auto mix = [&](uint32_t v) { for (int i = 0; i < 4; ++i) { h ^= (v >> (8 * i)) & 0xffu; h *= 0x100000001b3ull; } };
  mix((uint32_t)code.size());
  for (uint32_t v : code) mix(v);
  mix((uint32_t)rot.size());
  for (int32_t v : rot) mix((uint32_t)v);
  return h;
}

// ------------------------------------------------------------------------------------------------------
struct ParamsImpl {
  uint32_t k = 0, n = 0;
  int curve = 0;
  DevBuf g_w_u;         // n + 2 affine points: g || w || u
  DevBuf gl_w;          // n + 1 affine points: g_lagrange || w
  FixedBase fb_g, fb_gl;
  bool use_tables = true;   // k <= 19: fixed-base window tables; k >= 20 (or BZ_FORCE_GENERAL_MSM=1): bucket MSM over the raw bases
};

// The n_msm commitments of one call over the basis of p: g || w || u, or g_lagrange || w when `lagrange`.  MSM m sums
// d_main[m][0 .. p.n) and d_extra[m][0 .. npts - p.n) (the blind, and over g the U term) against that basis; d_main / d_extra
// are DEVICE arrays of device pointers.  d_out: n_msm affine points (64 B each), or with `xyzz_out` the table MSM's
// unnormalised XYZZ sums (128 B each).  The bucket path only returns affine points and rejects `xyzz_out`.  Stream-ordered
// on C->stream; its only allocation is the context's Jacobian scratch, grown as needed.
void params_commit_run(Ctx* C, const ParamsImpl& p, bool lagrange, const void* const* d_main, const void* const* d_extra,
                       uint32_t n_msm, void* d_out, bool xyzz_out = false);
// Copies the host pointer arrays into d (grown as needed) as [main... | extra...]; returns the device array (extras at + main.size())
const void* const* upload_msm_ptrs(Ctx* C, DevBuf& d, const std::vector<void*>& mainp, const std::vector<void*>& extrap);


struct CircuitCopy {
  uint32_t k, G, F, I, degree, bf;
  std::vector<std::pair<int, int>> aq, fq, iq;
  std::vector<std::pair<uint32_t, uint32_t>> perm;
  std::vector<HFe> consts;
  std::vector<Token> tokens;
  std::vector<uint32_t> gate_off;
  struct Lookup { std::vector<std::pair<uint32_t, uint32_t>> inputs, tables; };   // token ranges
  std::vector<Lookup> lookups;
  HFe vk_repr;
};

// kinds of the Regions table (see poly.cuh)
enum { R_VAL = 0, R_POLY = 1, R_MISC = 2, R_RANDPOLY = 3, R_SPOLY = 4, R_SHPOLY = 5, R_SHVAL = 6, R_HCOEF = 7 };

// commitment ids of the multiopen queries (instance / advice / permutation z / lookup (A', S', Z) / fixed / sigma / h / random)
enum { cid_inst = 0, cid_adv = 100000, cid_pz = 200000, cid_lk = 300000, cid_fix = 400000, cid_sig = 500000, cid_h = 600000, cid_rand = 600001 };
struct Query { int cid; int rot; PolyRef poly; int blind_kind; int blind_idx; int eval_idx; };   // eval_idx: position among the proof's evaluations (-1: h, computed by the verifier)   // blind_kind: 0 = one, 1 = per-proof blind slot

// The verifying key: what halo2's VerifyingKey holds (domain, constraint system, fixed and permutation commitments, and in
// cs.vk_repr the scalar vk.hash_into absorbs) plus the shape and multiopen layout derived from it.  Everything Verifier::run
// reads, and nothing else: building one allocates no device memory.
struct VkImpl {
  ParamsImpl* params = nullptr;
  CircuitCopy cs;
  uint32_t n = 0, qdeg = 0;
  uint32_t M = 0, L = 0, nsets = 0, chunk_len = 0, usable = 0;
  HFe omega, omega_inv;
  std::vector<uint64_t> vk_fixed_comm, vk_perm_comm;   // keygen_vk: commit_lagrange(column, Blind::default()) as affine (8 x u64 each)
  // static multiopen structure
  std::vector<Query> queries;
  struct CommInfo { PolyRef poly; int blind_kind, blind_idx; int set; int cid; };
  std::vector<CommInfo> cmap;                  // first-appearance order
  std::vector<std::vector<int>> point_sets;    // rotations per set, ordered by point index
  uint32_t nev = 0;                            // evaluations the proof carries (steps 14-18)
  uint32_t proof_size = 0;
  // slots
  uint32_t slot_inst(uint32_t i) const { return cs.G + i; }
  uint32_t slot_lk(uint32_t l, uint32_t which) const { return cs.G + cs.I + 3 * l + which; }   // 0 A', 1 S', 2 Z
  uint32_t slot_pz(uint32_t s) const { return cs.G + cs.I + 3 * L + s; }
  uint32_t misc_h() const { return 2 * L; }    // MISC slot of h(X), after the 2L compressed lookup expressions
  DevBuf vwork[16];      // verifier staging, kept across verify calls (no cudaMalloc / cudaFree per call)
};

// The shape part of keygen: circuit copy, domain constants, queries, multiopen structure, evaluation count and proof size.
// Host only; no GPU needed.
void vk_host_setup(const bzh::Field& F, VkImpl& vk, const bz_circuit* cin);

struct PkImpl : VkImpl {
  uint32_t ext_k = 0, ext_n = 0;
  uint32_t NS = 0, NC = 0;
  HFe ext_omega;
  // device images
  DevBuf lval;        // [F + M][n]  fixed values then sigma values (Lagrange)
  DevBuf shpoly;      // [F + M][n]  coefficient form
  DevBuf shcoset;     // [F + M + 5][ext_n]: fixed, sigma, l0, l_blind, l_last, active, coset_x
  DevBuf omega_pows;  // [n]
  DevBuf tev;         // [2^(ext_k-k)]
  // programs
  static constexpr uint32_t Q_TIERS = 3;     // h(X) tier t: terms whose quotient fits ext_n >> t points, evaluated on every 2^t-th extended point
  DevBuf lk_code, lk_rot, q_code[Q_TIERS], q_rot[Q_TIERS];
  uint32_t lk_ninstr = 0, q_ninstr[Q_TIERS] = {0, 0, 0}, q_muls[Q_TIERS] = {0, 0, 0};
  std::vector<uint32_t> h_lk_code, h_q_code[Q_TIERS];      // host copies (the programs are compiled without a GPU)
  std::vector<int32_t> h_lk_rot, h_q_rot[Q_TIERS];
  QuotientLaunchFn q_gen[Q_TIERS] = {nullptr, nullptr, nullptr};   // circuit-specialised straight-line kernel of the tier (gen_quotient.cu), or null: interpreter
  uint32_t n_exprs = 0;       // number of y-folded expressions E (gate polys, permutation, lookup terms)
  // Gate polynomials as h(X) evaluates them: every maximal sub-expression over fixed columns and constants only that contains
  // a product (after keygen's selector compression: q * prod_{i != r} (i - q), up to 8 multiplications per use) is evaluated
  // ONCE per proving key on the extended coset and kept as a derived shared column (shcoset slot F + M + 5 + j); the gate
  // polynomial queries it like a fixed column.  Same values at every point, so h(X) is unchanged.
  std::vector<DerivedColumn> derived;
  std::vector<Token> qtokens;
  std::vector<uint32_t> qgate_off;
  // const table layout
  uint32_t C_ONE, C_THETA, C_BETA, C_GAMMA, C_Y, C_X, C_XN, C_X1, C_X2, C_X3, C_X4, C_XI, C_Z, C_U, C_UINV, C_BD0, C_ROT0, C_YP0, cstride;
  std::vector<int> rots;                 // distinct rotations of all queries (+1, -1, last)
  std::map<int, uint32_t> rot_const;     // rotation -> const index of x * omega^rot
  // randomness layout (indices into the per-proof draw stream)
  uint32_t R = 0;
  uint32_t r_adv_rows, r_adv_blind, r_lk0, r_perm0, r_lkz0, r_randpoly, r_rand_blind, r_hblind, r_qprime, r_spoly, r_sblind, r_ipa;
  // per-proof blind slots (host)
  uint32_t nblinds = 0;
  // evaluation list (write order; nev entries)
  std::vector<EvalQuery> evals;
  DevBuf d_evals;
  // MISC slots
  uint32_t NM = 0, m_cin0, m_hpoly, m_qset0, m_qtmp0, m_qprime, m_ppoly, m_pprime, m_b, m_coef, m_scl, m_scr;
  // workspace cache
  struct Work {
    uint32_t batch = 0;
    DevBuf val, poly, coset, misc, rnd, wide, seeds, hext, hcoef, hext_low, hcoef_low, nd, consts, extras, evalout, commits, ptrs, descs, msm_jac, ipa_coefq, ipa_gm, ipa_tmp, lk_sorted, lk_err, scan_tmp, eval_tmp;
    void* h_pinned = nullptr; size_t h_pinned_bytes = 0;
    uint32_t* h_err = nullptr;      // pinned: error word of the device lookup permutation
  } work;
  ~PkImpl() { if (work.h_pinned) cudaFreeHost(work.h_pinned); if (work.h_err) cudaFreeHost(work.h_err); }
};

// Montgomery's trick on the host: v[i] <- 1 / v[i] (zeros stay zero), one field inversion for the whole vector
static inline void host_batch_invert(const bzh::Field& F, std::vector<HFe>& v) {
  std::vector<HFe> pre(v.size());
  HFe acc = F.one();
  for (size_t i = 0; i < v.size(); ++i) { pre[i] = acc; if (!v[i].is_zero()) acc = F.mul(acc, v[i]); }
  HFe inv = F.inv(acc);
  for (size_t i = v.size(); i-- > 0;) {
    if (v[i].is_zero()) continue;
    const HFe t = F.mul(inv, pre[i]);
    inv = F.mul(inv, v[i]);
    v[i] = t;
  }
}

struct HostPoint { uint8_t x[32], y[32]; bool identity; };

static inline void affine_to_host(const bzh::Field& Fq, const uint64_t* mont, HostPoint& p) {
  HFe x, y; memcpy(x.l, mont, 32); memcpy(y.l, mont + 4, 32);
  p.identity = x.is_zero() && y.is_zero();
  Fq.to_repr(x, p.x); Fq.to_repr(y, p.y);
}

struct ProofState {
  bzh::Blake2b st{"Halo2-Transcript"};
  uint8_t* out; size_t pos = 0;
  std::vector<HFe> blinds;      // per-proof blind slots
  std::vector<HFe> consts;      // per-proof const table (host copy)
  const uint8_t* wide;         // this proof's RNG words
};

static inline void t_common_scalar(ProofState& ps, const bzh::Field& F, const HFe& s) {
  uint8_t tag = 2, r[32]; F.to_repr(s, r); ps.st.update(&tag, 1); ps.st.update(r, 32);
}
static inline void t_write_scalar(ProofState& ps, const bzh::Field& F, const HFe& s) {
  uint8_t tag = 2, r[32]; F.to_repr(s, r); ps.st.update(&tag, 1); ps.st.update(r, 32);
  memcpy(ps.out + ps.pos, r, 32); ps.pos += 32;
}
static inline void t_common_point(ProofState& ps, const HostPoint& p) {
  if (p.identity) throw Error(BZ_ERR_INVALID, "cannot write points at infinity to the transcript");
  uint8_t tag = 1; ps.st.update(&tag, 1); ps.st.update(p.x, 32); ps.st.update(p.y, 32);
}
static inline void t_write_point(ProofState& ps, const HostPoint& p) {
  t_common_point(ps, p);
  memcpy(ps.out + ps.pos, p.x, 32);
  ps.out[ps.pos + 31] |= (uint8_t)((p.y[0] & 1) << 7);
  ps.pos += 32;
}
static inline HFe t_squeeze(ProofState& ps, const bzh::Field& F) {
  uint8_t tag = 0, h[64]; ps.st.update(&tag, 1); ps.st.finalize(h);
  return F.from_bytes_wide(h);
}
static inline HFe rnd_host(const ProofState& ps, const bzh::Field& F, uint32_t idx) { return F.from_bytes_wide(ps.wide + (size_t)idx * 64); }

}  // namespace bz

struct bz_params { bz::ParamsImpl p; };
struct bz_pk { bz::PkImpl p; };
struct bz_vk { bz::VkImpl v; };
static inline bz::Ctx* ctx_of(bz_ctx* c) { return &c->c; }

#define PV_TRY(ctx_, ...)                                     \
  if (!(ctx_)) return BZ_ERR_INVALID;                         \
  bz::Ctx* C = ctx_of(ctx_);                                  \
  try {                                                       \
    cudaSetDevice(C->device);                                 \
    __VA_ARGS__;                                              \
    return BZ_OK;                                             \
  } catch (const bz::Error& e) {                              \
    C->last_error = e.what();                                 \
    return e.code;                                            \
  } catch (const std::exception& e) {                         \
    C->last_error = e.what();                                 \
    return BZ_ERR_INVALID;                                    \
  }

#define API __attribute__((visibility("default")))

