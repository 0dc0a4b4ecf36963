// Device kernels of the prover's polynomial layer (everything between the NTTs and the MSMs):
// expression interpreter (lookup compression on the Lagrange domain, h(X) on the extended coset),
// grand-product scans, Horner evaluation, multiopen accumulation / synthetic division, IPA folding.
// Replaces the loops of halo2_proofs 0.2.0 src/poly/evaluator.rs, src/plonk/{permutation,lookup,vanishing}/
// prover.rs, src/arithmetic.rs::{eval_polynomial, kate_division, compute_inner_product},
// src/poly/multiopen/prover.rs, src/poly/commitment/prover.rs  (SURVEY §8 a6-a11).
//
// Batch-major: every kernel processes the same step of B independent proofs (blockIdx.y / .z = proof),
// per-proof challenges live in a device scalar table `sc[b][*]`.
#pragma once
#include "field.cuh"
#include "evalprog.h"

namespace bz {

// A polynomial / column lives at  base[kind] + b * stride[kind] + slot * len ; kind indexes this table.
struct Regions {
  void* base[8];
  uint64_t stride[8];     // elements per proof (0 = shared across the batch)
};
struct PolyRef { uint32_t kind, slot; };

template <class P> __device__ __forceinline__ Fe<P>* region_ptr(const Regions& r, PolyRef ref, uint32_t b, uint64_t len) {
  return reinterpret_cast<Fe<P>*>(r.base[ref.kind]) + (uint64_t)b * r.stride[ref.kind] + (uint64_t)ref.slot * len;
}

// ---- interpreter ---------------------------------------------------------------------------------
// opcodes, EVAL_STACK / EVAL_TMP and the host-side program builder: evalprog.h

template <class P> struct EvalArgs {
  const uint32_t* code;
  uint32_t n_instr;
  uint32_t logN;                 // domain size 2^logN
  const int32_t* rot;            // rotation table: element offsets (already scaled for the domain)
  const Fe<P>* pbase;            // per-proof arrays: pbase + b*pstride + slot*N
  uint64_t pstride;
  const Fe<P>* sbase;            // shared arrays:    sbase + slot*N
  const Fe<P>* consts;           // per-proof constants: consts + b*cstride
  uint32_t cstride;
  Fe<P>* out;                    // outputs: out + b*ostride + k*N
  uint64_t ostride;
  const Fe<P>* tev;              // t_evaluations (for OP_MUL_T_STORE), length tn (power of two)
  uint32_t tn;
  uint32_t stride_log;           // evaluate at domain points j = i << stride_log only (outputs stay dense, indexed by i)
  uint32_t first;                // this launch covers the points i >= first (one large proof across GPUs: every rank a range)
};

template <class P>
__global__ void __launch_bounds__(128) eval_program_kernel(const __grid_constant__ EvalArgs<P> a) {
  extern __shared__ uint32_t s_code[];
  for (uint32_t t = threadIdx.x; t < a.n_instr; t += blockDim.x) s_code[t] = a.code[t];
  __syncthreads();
  const uint32_t N = 1u << a.logN;
  const uint32_t i = a.first + blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t b = blockIdx.y;
  if (i >= (N >> a.stride_log)) return;
  const uint32_t jp = i << a.stride_log;         // the domain point this thread evaluates
  const Fe<P>* pb = a.pbase + (uint64_t)b * a.pstride;
  const Fe<P>* cb = a.consts + (uint64_t)b * a.cstride;
  Fe<P> st[EVAL_STACK];
  Fe<P> tmp[EVAL_TMP];           // shared sub-expressions of the gate DAG (evalprog.h)
  Fe<P> acc = fe_zero<P>();
  int sp = 0;
  for (uint32_t pc = 0; pc < a.n_instr; ++pc) {
    const uint32_t ins = s_code[pc];
    const uint32_t op = ins & 15u, x = (ins >> 4) & 0xfffu, y = ins >> 16;
    switch (op) {
      case OP_PUSH_P: { uint32_t idx = (jp + (uint32_t)a.rot[y]) & (N - 1); st[sp++] = fe_load(pb + ((uint64_t)x << a.logN) + idx); break; }
      case OP_PUSH_S: { uint32_t idx = (jp + (uint32_t)a.rot[y]) & (N - 1); st[sp++] = fe_load(a.sbase + ((uint64_t)x << a.logN) + idx); break; }
      case OP_PUSH_C: st[sp++] = fe_load(cb + (ins >> 4)); break;
      case OP_ADD: --sp; st[sp - 1] = fe_add(st[sp - 1], st[sp]); break;
      case OP_SUB: --sp; st[sp - 1] = fe_sub(st[sp - 1], st[sp]); break;
      case OP_MUL: --sp; st[sp - 1] = fe_mul(st[sp - 1], st[sp]); break;
      case OP_NEG: st[sp - 1] = fe_neg(st[sp - 1]); break;
      case OP_MULC: st[sp - 1] = fe_mul(st[sp - 1], fe_load(cb + (ins >> 4))); break;
      case OP_ADDC: st[sp - 1] = fe_add(st[sp - 1], fe_load(cb + (ins >> 4))); break;
      case OP_FOLD: --sp; acc = fe_add(fe_mul(acc, fe_load(cb + (ins >> 4))), st[sp]); break;
      case OP_STORE: --sp; fe_store(a.out + (uint64_t)b * a.ostride + ((uint64_t)(ins >> 4) << a.logN) + i, st[sp]); break;
      case OP_ACC_MULC: acc = fe_mul(acc, fe_load(cb + (ins >> 4))); break;
      case OP_MUL_T_STORE: fe_store(a.out + (uint64_t)b * a.ostride + i, fe_mul(acc, fe_load(a.tev + (jp & (a.tn - 1))))); break;
      case OP_TEE: tmp[ins >> 4] = st[sp - 1]; break;
      case OP_PUSH_T: st[sp++] = tmp[ins >> 4]; break;
      default: break;
    }
  }
}

// dst[b][i] += src[b][i]  (i < count): the low-degree part of h(X), interpolated on the half-size coset, joins the rest
template <class P>
__global__ void add_low_kernel(Fe<P>* __restrict__ dst, uint64_t dst_stride, const Fe<P>* __restrict__ src, uint32_t count) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (i >= count) return;
  Fe<P>* d = dst + (uint64_t)b * dst_stride + i;
  fe_store(d, fe_add(fe_load(d), fe_load(src + (uint64_t)b * count + i)));
}

// ---- 512-bit RNG words -> field elements (pasta Field::random = from_u512) --------------------------
template <class P>
__global__ void from_u512_kernel(const uint32_t* __restrict__ wide, Fe<P>* __restrict__ out, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t w[16];
  const uint4* q = reinterpret_cast<const uint4*>(wide + i * 16);
#pragma unroll
  for (int j = 0; j < 4; ++j) { uint4 v = q[j]; w[4 * j] = v.x; w[4 * j + 1] = v.y; w[4 * j + 2] = v.z; w[4 * j + 3] = v.w; }
  fe_store(out + i, fe_from_u512<P>(w));
}

// dst[b][dst_off + j] = src[b][src_off + j]  for a list of (dst region/slot/offset, src offset, count) copies
struct CopyDesc { PolyRef dst; uint32_t dst_off; uint32_t src_off; uint32_t count; };
template <class P>
__global__ void copy_rows_kernel(Regions reg, uint64_t len, const CopyDesc* __restrict__ descs, const Fe<P>* __restrict__ src, uint64_t src_stride) {
  const CopyDesc d = descs[blockIdx.x];
  const uint32_t b = blockIdx.y;
  Fe<P>* dst = region_ptr<P>(reg, d.dst, b, len) + d.dst_off;
  const Fe<P>* s = src + (uint64_t)b * src_stride + d.src_off;
  for (uint32_t j = threadIdx.x; j < d.count; j += blockDim.x) fe_store(dst + j, fe_load(s + j));
}

// ---- lookup permutation (U: halo2_proofs 0.2.0 src/plonk/lookup/prover.rs::permute_expression_pair) -------------
// One CTA per (lookup, proof).  The reference sorts the compressed input expression over the usable rows (Ord = the
// canonical integer), keeps a BTreeMap multiset of the table expression, writes the table value next to the FIRST row of
// every run of equal inputs and fills the remaining ("repeated") rows, last row first, with the left-over table values
// in ascending order.  Here: two shared-memory bitonic sorts of 256-bit canonical keys, one binary search per distinct
// input value, two block scans and a gather -- results are the same canonical values, hence bit-identical columns.
struct LookupPermDesc { PolyRef cin, ctab, aout, sout; };
constexpr int LKP_THREADS = 1024;
constexpr uint32_t LKP_MAX_N = 4096;         // 44 B of shared memory per row
inline size_t lookup_permute_smem(uint32_t n) { return (size_t)n * 32 + (size_t)3 * n * 4; }

__device__ __forceinline__ bool key_less(const uint4& a0, const uint4& a1, const uint4& b0, const uint4& b1) {
  sub_cc(a0.x, b0.x); subc_cc(a0.y, b0.y); subc_cc(a0.z, b0.z); subc_cc(a0.w, b0.w);
  subc_cc(a1.x, b1.x); subc_cc(a1.y, b1.y); subc_cc(a1.z, b1.z); subc_cc(a1.w, b1.w);
  return subc(0u, 0u) != 0u;             // borrow out  <=>  a < b
}
__device__ __forceinline__ bool key_eq(const uint4& a0, const uint4& a1, const uint4& b0, const uint4& b1) {
  return ((a0.x ^ b0.x) | (a0.y ^ b0.y) | (a0.z ^ b0.z) | (a0.w ^ b0.w) | (a1.x ^ b1.x) | (a1.y ^ b1.y) | (a1.z ^ b1.z) | (a1.w ^ b1.w)) == 0u;
}
// ascending bitonic sort of npad (power of two) keys in shared memory, K[2i], K[2i+1] = low / high half of key i
__device__ __forceinline__ void bitonic_sort_keys(uint4* K, uint32_t npad) {
  for (uint32_t k = 2; k <= npad; k <<= 1)
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < (npad >> 1); t += blockDim.x) {
        const uint32_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1)), p = i | j;
        const uint4 a0 = K[2 * i], a1 = K[2 * i + 1], b0 = K[2 * p], b1 = K[2 * p + 1];
        const bool up = (i & k) == 0;
        const bool sw = up ? key_less(b0, b1, a0, a1) : key_less(a0, a1, b0, b1);
        if (sw) { K[2 * i] = b0; K[2 * i + 1] = b1; K[2 * p] = a0; K[2 * p + 1] = a1; }
      }
      __syncthreads();
    }
}
// in-place exclusive prefix sum of arr[0..len) by the whole CTA; returns the total.  wsum: 33 words of shared memory
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t* arr, uint32_t len, uint32_t* wsum) {
  const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
  const uint32_t per = (len + blockDim.x - 1) / blockDim.x, lo = min(tid * per, len), hi = min(lo + per, len);
  uint32_t s = 0;
  for (uint32_t i = lo; i < hi; ++i) s += arr[i];
  uint32_t incl = s;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { uint32_t o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= (uint32_t)d) incl += o; }
  if (lane == 31) wsum[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    uint32_t v = lane < nw ? wsum[lane] : 0u, iv = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t o = __shfl_up_sync(0xffffffffu, iv, d); if (lane >= (uint32_t)d) iv += o; }
    if (lane < nw) wsum[lane] = iv - v;
    if (lane == 31) wsum[32] = iv;
  }
  __syncthreads();
  uint32_t run = wsum[wid] + incl - s;
  for (uint32_t i = lo; i < hi; ++i) { uint32_t v = arr[i]; arr[i] = run; run += v; }
  const uint32_t total = wsum[32];
  __syncthreads();
  return total;
}

template <class P>
__global__ void __launch_bounds__(LKP_THREADS) lookup_permute_kernel(Regions reg, uint32_t n, uint32_t usable, const LookupPermDesc* __restrict__ descs,
                                      Fe<P>* __restrict__ tsorted /* [proof][lookup][n] canonical */, uint32_t* __restrict__ err) {
  extern __shared__ uint4 lkp_smem[];
  __shared__ uint32_t wsum[33];
  uint4* K = lkp_smem;
  uint32_t* removed = reinterpret_cast<uint32_t*>(lkp_smem + 2 * (size_t)n);     // -> rank among the left-over table rows
  uint32_t* repeat = removed + n;                                                // -> rank among the repeated input rows
  uint32_t* left = repeat + n;                                                   // left-over table rows, ascending
  const uint32_t l = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const LookupPermDesc d = descs[l];
  Fe<P>* T = tsorted + ((uint64_t)b * gridDim.x + l) * n;
  const uint4 ff = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
  auto load_keys = [&](PolyRef src) {
    const Fe<P>* s = region_ptr<P>(reg, src, b, n);
    for (uint32_t i = tid; i < n; i += LKP_THREADS) {
      if (i < usable) {
        Fe<P> v = fe_from_mont(fe_load(s + i));
        K[2 * i] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]); K[2 * i + 1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
      } else { K[2 * i] = ff; K[2 * i + 1] = ff; }      // larger than every canonical value: stays behind the usable rows
    }
    __syncthreads();
  };
  // 1. table expression, sorted, canonical -> global scratch
  load_keys(d.ctab);
  bitonic_sort_keys(K, n);
  for (uint32_t i = tid; i < usable; i += LKP_THREADS) {
    uint4* o = reinterpret_cast<uint4*>(T + i);
    o[0] = K[2 * i]; o[1] = K[2 * i + 1];
  }
  __syncthreads();
  // 2. input expression, sorted: A'
  load_keys(d.cin);
  bitonic_sort_keys(K, n);
  Fe<P>* aout = region_ptr<P>(reg, d.aout, b, n);
  Fe<P>* sout = region_ptr<P>(reg, d.sout, b, n);
  for (uint32_t i = tid; i < n; i += LKP_THREADS) {
    removed[i] = 0;
    bool rep = false;
    if (i < usable) {
      const uint4 a0 = K[2 * i], a1 = K[2 * i + 1];
      Fe<P> v; v.l[0] = a0.x; v.l[1] = a0.y; v.l[2] = a0.z; v.l[3] = a0.w; v.l[4] = a1.x; v.l[5] = a1.y; v.l[6] = a1.z; v.l[7] = a1.w;
      fe_store(aout + i, fe_to_mont(v));
      rep = i > 0 && key_eq(a0, a1, K[2 * i - 2], K[2 * i - 1]);
    }
    repeat[i] = rep ? 1u : 0u;
  }
  __syncthreads();
  // 3. every distinct input value takes one copy out of the table multiset
  for (uint32_t i = tid; i < usable; i += LKP_THREADS) {
    if (repeat[i]) continue;
    const uint4 a0 = K[2 * i], a1 = K[2 * i + 1];
    uint32_t lo = 0, hi = usable;                       // lower_bound
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      const uint4* q = reinterpret_cast<const uint4*>(T + mid);
      if (key_less(q[0], q[1], a0, a1)) lo = mid + 1; else hi = mid;
    }
    bool ok = lo < usable;
    if (ok) { const uint4* q = reinterpret_cast<const uint4*>(T + lo); ok = key_eq(q[0], q[1], a0, a1); }
    if (ok) removed[lo] = 1; else atomicOr(err + b, 1u);    // Error::ConstraintSystemFailure: input not in the table (one error word per proof)
  }
  __syncthreads();
  for (uint32_t i = tid; i < n; i += LKP_THREADS) removed[i] = (i < usable && !removed[i]) ? 1u : 0u;    // now: "kept"
  __syncthreads();
  const uint32_t n_left = block_exclusive_scan(removed, n, wsum);
  for (uint32_t i = tid; i < usable; i += LKP_THREADS) {
    const uint32_t nxt = (i + 1 < n) ? removed[i + 1] : n_left;
    if (nxt != removed[i]) left[removed[i]] = i;
  }
  __syncthreads();
  const uint32_t n_rep = block_exclusive_scan(repeat, n, wsum);
  if (n_rep != n_left) { if (tid == 0) atomicOr(err + b, 2u); return; }
  // 4. S'
  for (uint32_t i = tid; i < usable; i += LKP_THREADS) {
    const uint32_t nxt = (i + 1 < n) ? repeat[i + 1] : n_rep;
    Fe<P> v;
    if (nxt == repeat[i]) {
      const uint4 a0 = K[2 * i], a1 = K[2 * i + 1];
      v.l[0] = a0.x; v.l[1] = a0.y; v.l[2] = a0.z; v.l[3] = a0.w; v.l[4] = a1.x; v.l[5] = a1.y; v.l[6] = a1.z; v.l[7] = a1.w;
    } else {
      v = fe_load(T + left[n_left - 1 - repeat[i]]);
    }
    fe_store(sout + i, fe_to_mont(v));
  }
}

// ---- grand products ----------------------------------------------------------------------------------
// halo2 multiplies every numerator by batch_invert(den), which leaves the inverse of a zero denominator at zero, so
// z[i+1] = z[i] * num[i] * inv0(den[i]) drops to 0 after a zero denominator and is unaffected before it.  The fraction
// kernels store such a row as (num, den) = (0, 1): the term is the same, and every suffix product of den stays non-zero,
// which the finish kernels (z[i] = z0 * pnum[i] * sden[i] / sden[0]) need.
// permutation fractions for one column set: num[i] = prod_j (v_j + (beta delta^j) w^i + gamma),
//                                            den[i] = prod_j (v_j + beta sigma_j + gamma)
struct PermSetDesc { uint32_t ncols; uint32_t val_kind[8]; uint32_t val_slot[8]; uint32_t sigma_slot[8]; uint32_t bd_const[8]; };
template <class P>
__global__ void perm_fraction_kernel(Regions reg, uint32_t n, PermSetDesc d, const Fe<P>* __restrict__ sigma_vals /*shared [m][n]*/,
                                     const Fe<P>* __restrict__ omega_pows, const Fe<P>* __restrict__ consts, uint32_t cstride,
                                     uint32_t c_beta, uint32_t c_gamma, Fe<P>* __restrict__ num, Fe<P>* __restrict__ den, uint64_t nd_stride) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b = blockIdx.y;
  if (i >= n) return;
  const Fe<P>* cb = consts + (uint64_t)b * cstride;
  Fe<P> beta = fe_load(cb + c_beta), gamma = fe_load(cb + c_gamma);
  Fe<P> w = fe_load(omega_pows + i);
  Fe<P> nu = fe_one<P>(), de = fe_one<P>();
  for (uint32_t j = 0; j < d.ncols; ++j) {
    PolyRef ref{d.val_kind[j], d.val_slot[j]};
    Fe<P> v = fe_load(region_ptr<P>(reg, ref, b, n) + i);
    Fe<P> vg = fe_add(v, gamma);
    Fe<P> s = fe_load(sigma_vals + (uint64_t)d.sigma_slot[j] * n + i);
    de = fe_mul(de, fe_add(vg, fe_mul(beta, s)));
    nu = fe_mul(nu, fe_add(vg, fe_mul(fe_load(cb + d.bd_const[j]), w)));
  }
  if (fe_is_zero(de)) { nu = fe_zero<P>(); de = fe_one<P>(); }
  fe_store(num + (uint64_t)b * nd_stride + i, nu);
  fe_store(den + (uint64_t)b * nd_stride + i, de);
}

// lookup fractions: num = (cin + beta)(ctab + gamma), den = (a' + beta)(s' + gamma)
template <class P>
__global__ void lookup_fraction_kernel(Regions reg, uint32_t n, PolyRef cin, PolyRef ctab, PolyRef ap, PolyRef sp,
                                       const Fe<P>* __restrict__ consts, uint32_t cstride, uint32_t c_beta, uint32_t c_gamma,
                                       Fe<P>* __restrict__ num, Fe<P>* __restrict__ den, uint64_t nd_stride) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b = blockIdx.y;
  if (i >= n) return;
  const Fe<P>* cb = consts + (uint64_t)b * cstride;
  Fe<P> beta = fe_load(cb + c_beta), gamma = fe_load(cb + c_gamma);
  Fe<P> nu = fe_mul(fe_add(fe_load(region_ptr<P>(reg, cin, b, n) + i), beta), fe_add(fe_load(region_ptr<P>(reg, ctab, b, n) + i), gamma));
  Fe<P> de = fe_mul(fe_add(fe_load(region_ptr<P>(reg, ap, b, n) + i), beta), fe_add(fe_load(region_ptr<P>(reg, sp, b, n) + i), gamma));
  if (fe_is_zero(de)) { nu = fe_zero<P>(); de = fe_one<P>(); }
  fe_store(num + (uint64_t)b * nd_stride + i, nu);
  fe_store(den + (uint64_t)b * nd_stride + i, de);
}

// warp-level inclusive scan with field multiplication; `rev` scans from the high lane down
template <class P> __device__ __forceinline__ Fe<P> warp_scan_mul(Fe<P> v, bool rev) {
  const uint32_t lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    Fe<P> o;
#pragma unroll
    for (int k = 0; k < 8; ++k) o.l[k] = rev ? __shfl_down_sync(0xffffffffu, v.l[k], d) : __shfl_up_sync(0xffffffffu, v.l[k], d);
    bool take = rev ? (lane + d < 32) : (lane >= (uint32_t)d);
    if (take) v = fe_mul(v, o);
  }
  return v;
}

// One CTA (256 threads) per proof scans a whole array tile by tile with a running carry.
//   mode 0: out[i] = prod_{t<i} in[t]   (exclusive prefix)      mode 1: out[i] = prod_{t>=i} in[t]  (inclusive suffix)
constexpr int SCAN_THREADS = 256, SCAN_PER = 8, SCAN_TILE = SCAN_THREADS * SCAN_PER;
// Large arrays (the scaled circuit) run it three times: CTA c of grid.x owns `tiles_per_cta` tiles -- pass 1 writes only the
// product of its tiles (totals_out), the same kernel then scans those totals (one tile), pass 3 rescans with the carry-in.
template <class P>
__global__ void __launch_bounds__(SCAN_THREADS) product_scan_kernel(const Fe<P>* __restrict__ in, Fe<P>* __restrict__ out, uint32_t n, uint64_t stride, int mode,
                                                                    uint32_t tiles_per_cta = 0xffffffffu, const Fe<P>* __restrict__ carry_in = nullptr,
                                                                    Fe<P>* __restrict__ totals_out = nullptr) {
  __shared__ Fe<P> warp_tot[SCAN_THREADS / 32];
  __shared__ Fe<P> carry_sh;
  const uint32_t b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const Fe<P>* src = in + (uint64_t)b * stride;
  Fe<P>* dst = out + (uint64_t)b * stride;
  const bool rev = mode == 1;
  Fe<P> carry = carry_in ? fe_load(carry_in + (uint64_t)b * gridDim.x + blockIdx.x) : fe_one<P>();
  const uint32_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  const uint32_t tile0 = tiles_per_cta == 0xffffffffu ? 0u : blockIdx.x * tiles_per_cta;
  const uint32_t tile1 = tiles_per_cta == 0xffffffffu ? ntiles : min(ntiles, tile0 + tiles_per_cta);
  for (uint32_t tile = tile0; tile < tile1; ++tile) {
    // element range of this thread inside the tile (in scan order)
    uint32_t base = tile * SCAN_TILE + tid * SCAN_PER;
    Fe<P> v[SCAN_PER];
    Fe<P> tot = fe_one<P>();
#pragma unroll
    for (int j = 0; j < SCAN_PER; ++j) {
      uint32_t pos = base + j;                       // position in scan order
      uint32_t idx = rev ? (n - 1 - pos) : pos;
      v[j] = pos < n ? fe_load(src + idx) : fe_one<P>();
      tot = fe_mul(tot, v[j]);
    }
    // in scan order "forward" always means increasing pos, so use the non-reversed warp scan
    Fe<P> incl = warp_scan_mul<P>(tot, false);
    if (lane == 31) warp_tot[wid] = incl;
    __syncthreads();
    // exclusive prefix over warps (8 warps: serial by every thread)
    Fe<P> wpre = fe_one<P>();
    for (uint32_t w = 0; w < wid; ++w) wpre = fe_mul(wpre, warp_tot[w]);
    // exclusive prefix for this thread = carry * wpre * (incl / tot)  -> recompute via shuffle of incl
    Fe<P> prev;
#pragma unroll
    for (int k = 0; k < 8; ++k) prev.l[k] = __shfl_up_sync(0xffffffffu, incl.l[k], 1);
    if (lane == 0) prev = fe_one<P>();
    Fe<P> run = fe_mul(fe_mul(carry, wpre), prev);
#pragma unroll
    for (int j = 0; j < SCAN_PER; ++j) {
      uint32_t pos = base + j;
      if (pos < n && !totals_out) {
        uint32_t idx = rev ? (n - 1 - pos) : pos;
        if (mode == 0) { fe_store(dst + idx, run); run = fe_mul(run, v[j]); }
        else { run = fe_mul(run, v[j]); fe_store(dst + idx, run); }
      }
    }
    // new carry = carry * product of the whole tile
    if (tid == SCAN_THREADS - 1) {
      Fe<P> t = fe_mul(fe_mul(carry, wpre), incl);
      carry_sh = t;
    }
    __syncthreads();
    carry = carry_sh;
    __syncthreads();
  }
  if (totals_out && tid == 0) fe_store(totals_out + (uint64_t)b * gridDim.x + blockIdx.x, carry);
}

// z[i] = z0 * pnum[i] * sden[i] / sden[0]   (z0: *z0_ptr[b * z0_stride] or 1 if null)
template <class P>
__global__ void grand_product_finish_kernel(const Fe<P>* __restrict__ pnum, const Fe<P>* __restrict__ sden, uint64_t nd_stride,
                                            Regions reg, PolyRef zref, uint32_t n, PolyRef z0ref, uint32_t z0_index, int has_z0) {
  __shared__ Fe<P> scale_sh;
  const uint32_t b = blockIdx.y;
  if (threadIdx.x == 0) {
    Fe<P> inv = fe_inv_gcd(fe_load(sden + (uint64_t)b * nd_stride));     // one lane, pure latency: binary GCD (ALU pipe) instead of a Fermat chain
    if (has_z0) inv = fe_mul(inv, fe_load(region_ptr<P>(reg, z0ref, b, n) + z0_index));
    scale_sh = inv;
  }
  __syncthreads();
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fe<P> v = fe_mul(fe_mul(fe_load(pnum + (uint64_t)b * nd_stride + i), fe_load(sden + (uint64_t)b * nd_stride + i)), scale_sh);
  fe_store(region_ptr<P>(reg, zref, b, n) + i, v);
}

// All grand products of a proof in one launch (blockIdx.z = product): the first `nsets` products are the permutation sets,
// chained through z_s[0] = z_{s-1}[u] (u = first unusable row); the others (lookups) start at 1.
//   z_g[i] = z0_g * pnum_g[i] * sden_g[i] / sden_g[0],   z0_s = prod_{s' < s} pnum_s'[u] * sden_s'[u] / sden_s'[0]
// The <= 8 inversions a product needs share one Fermat chain (Montgomery's trick; no sden is zero), so a batch pays the
// inversion latency once instead of once per product.  ONE CTA per (proof, product) walks all rows: B x G inversions per batch
// (launch site in prover.cu).
struct GpBatchDesc { uint32_t nprod, nsets; PolyRef zref[8]; };
template <class P>
__global__ void grand_product_finish_batch_kernel(const Fe<P>* __restrict__ pnum, const Fe<P>* __restrict__ sden, uint64_t prod_stride, uint64_t nd_stride,
                                                  Regions reg, GpBatchDesc d, uint32_t n, uint32_t u) {
  __shared__ Fe<P> scale_sh;
  const uint32_t b = blockIdx.y, g = blockIdx.z;
  if (threadIdx.x == 0) {
    const uint32_t g0 = g < d.nsets ? 0u : g;
    Fe<P> pre[8], s0[8];
    Fe<P> acc = fe_one<P>();
    for (uint32_t gp = g0; gp <= g; ++gp) {
      s0[gp - g0] = fe_load(sden + (uint64_t)gp * prod_stride + (uint64_t)b * nd_stride);
      pre[gp - g0] = acc;
      acc = fe_mul(acc, s0[gp - g0]);
    }
    Fe<P> inv = fe_inv_gcd(acc);
    Fe<P> z0 = fe_one<P>(), mine = fe_zero<P>();
    for (uint32_t gp = g + 1; gp-- > g0;) {                       // 1 / sden_gp[0], last product first
      const Fe<P> iv = fe_mul(inv, pre[gp - g0]);
      inv = fe_mul(inv, s0[gp - g0]);
      if (gp == g) mine = iv;
      else {
        const uint64_t at = (uint64_t)gp * prod_stride + (uint64_t)b * nd_stride + u;
        z0 = fe_mul(z0, fe_mul(fe_mul(fe_load(pnum + at), fe_load(sden + at)), iv));
      }
    }
    scale_sh = fe_mul(z0, mine);
  }
  __syncthreads();
  const Fe<P> scale = scale_sh;
  for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
    const uint64_t at = (uint64_t)g * prod_stride + (uint64_t)b * nd_stride + i;
    fe_store(region_ptr<P>(reg, d.zref[g], b, n) + i, fe_mul(fe_mul(fe_load(pnum + at), fe_load(sden + at)), scale));
  }
}

// ---- Horner evaluation: one CTA per (query, proof) ---------------------------------------------------
struct EvalQuery { PolyRef poly; uint32_t point_const; };     // point = consts[b][point_const]
constexpr int EVALQ_THREADS = 128;
// Large polynomials: gridDim.z CTAs per (query, proof), each over a contiguous slice; the slice sums go to `out` at
// [(b * out_stride + qi) * gridDim.z + z] and eval_reduce_kernel adds them.
template <class P>
__global__ void __launch_bounds__(EVALQ_THREADS) eval_queries_kernel(Regions reg, uint32_t n, const EvalQuery* __restrict__ queries,
                                    const Fe<P>* __restrict__ consts, uint32_t cstride, Fe<P>* __restrict__ out, uint32_t out_stride) {
  __shared__ Fe<P> sh[EVALQ_THREADS];
  const uint32_t qi = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const EvalQuery q = queries[qi];
  const Fe<P>* poly = region_ptr<P>(reg, q.poly, b, n);
  const Fe<P> x = fe_load(consts + (uint64_t)b * cstride + q.point_const);
  const uint32_t slice = (n + gridDim.z - 1) / gridDim.z, s_lo = min(blockIdx.z * slice, n), s_hi = min(s_lo + slice, n);
  const uint32_t len = (s_hi - s_lo + EVALQ_THREADS - 1) / EVALQ_THREADS;
  const uint32_t lo = min(s_lo + tid * len, s_hi), hi = min(lo + len, s_hi);
  Fe<P> acc = fe_zero<P>();
  for (uint32_t i = hi; i > lo; --i) acc = fe_add(fe_mul(acc, x), fe_load(poly + i - 1));
  if (lo < hi && lo > 0) acc = fe_mul(acc, fe_pow_u64<P>(x, lo));
  sh[tid] = (lo < hi) ? acc : fe_zero<P>();
  __syncthreads();
  for (uint32_t d = EVALQ_THREADS >> 1; d > 0; d >>= 1) {
    if (tid < d) sh[tid] = fe_add(sh[tid], sh[tid + d]);
    __syncthreads();
  }
  if (tid == 0) fe_store(out + ((uint64_t)b * out_stride + qi) * gridDim.z + blockIdx.z, sh[0]);
}
// out[i] = sum of the `splits` slice sums of evaluation i
template <class P>
__global__ void eval_reduce_kernel(const Fe<P>* __restrict__ partial, uint32_t splits, Fe<P>* __restrict__ out, uint32_t count) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  Fe<P> acc = fe_zero<P>();
  for (uint32_t z = 0; z < splits; ++z) acc = fe_add(acc, fe_load(partial + (uint64_t)i * splits + z));
  fe_store(out + i, acc);
}

// ---- out[i] = Horner_j( polys[j][i] ; x ) = ((p0 x + p1) x + p2) ...   (multiopen / vanishing / IPA combos) ----
struct LinCombDesc { PolyRef out; uint32_t x_const; uint32_t count; uint32_t first; };   // polys = refs[first .. first+count)
template <class P>
__global__ void lincomb_kernel(Regions reg, uint32_t n, const LinCombDesc* __restrict__ descs, const PolyRef* __restrict__ refs,
                               const Fe<P>* __restrict__ consts, uint32_t cstride) {
  const LinCombDesc d = descs[blockIdx.z];
  const uint32_t b = blockIdx.y;
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Fe<P> x = fe_load(consts + (uint64_t)b * cstride + d.x_const);
  Fe<P> acc = fe_load(region_ptr<P>(reg, refs[d.first], b, n) + i);
  for (uint32_t j = 1; j < d.count; ++j)
    acc = fe_add(fe_mul(acc, x), fe_load(region_ptr<P>(reg, refs[d.first + j], b, n) + i));
  fe_store(region_ptr<P>(reg, d.out, b, n) + i, acc);
}

// ---- kate_division: q(X) = floor(a(X) / (X - pt)), q has n-1 coefficients, q[n-1] := 0 -----------------
// One CTA per (division, proof).  r[i] = a[i+1] + pt * r[i+1]; chunks per thread + log-step scan of the
// chunk transfer maps r[lo] = L + pt^len * r[hi].
constexpr int KATE_THREADS = 256;
struct KateDesc { PolyRef in, out; uint32_t point_const; };
// Large polynomials: gridDim.z CTAs per (division, proof), CTA z over the contiguous slice [z*slice, (z+1)*slice).  Pass 1
// (totals_out != null) only reports r[slice_lo] under a zero carry-in; kate_carry_kernel chains the slices from the top;
// pass 2 (carry_in != null) redoes the slice with its true carry-in r[slice_hi] and writes the quotient.
template <class P>
__global__ void __launch_bounds__(KATE_THREADS) kate_division_kernel(Regions reg, uint32_t n, const KateDesc* __restrict__ descs,
                                     const Fe<P>* __restrict__ consts, uint32_t cstride,
                                     const Fe<P>* __restrict__ carry_in = nullptr, Fe<P>* __restrict__ totals_out = nullptr) {
  __shared__ Fe<P> sh[2][KATE_THREADS + 1];
  const KateDesc d = descs[blockIdx.x];
  const uint32_t b = blockIdx.y, tid = threadIdx.x;
  const Fe<P>* a = region_ptr<P>(reg, d.in, b, n);
  Fe<P>* q = region_ptr<P>(reg, d.out, b, n);
  const Fe<P> pt = fe_load(consts + (uint64_t)b * cstride + d.point_const);
  const uint32_t slice = (n + gridDim.z - 1) / gridDim.z, s_lo = min(blockIdx.z * slice, n), s_hi = min(s_lo + slice, n);
  const uint64_t slot = ((uint64_t)b * gridDim.x + blockIdx.x) * gridDim.z + blockIdx.z;
  const uint32_t len = (s_hi - s_lo + KATE_THREADS - 1) / KATE_THREADS;
  const uint32_t lo = min(s_lo + tid * len, s_hi), hi = min(lo + len, s_hi);
  // local pass with zero carry-in
  Fe<P> r = fe_zero<P>();
  for (uint32_t i = hi; i > lo; --i) {
    Fe<P> ai = (i < n) ? fe_load(a + i) : fe_zero<P>();        // a[i] with a[n] = 0
    r = fe_add(ai, fe_mul(pt, r));                              // r[i-1]
  }
  // suffix scan over threads: R_t = L_t + B * R_{t+1},  B = pt^len   (threads with empty chunks: L = 0, act as identity*B)
  Fe<P> Bp = fe_pow_u64<P>(pt, len);
  int cur = 0;
  sh[0][tid] = r;
  if (tid == 0) { sh[0][KATE_THREADS] = fe_zero<P>(); sh[1][KATE_THREADS] = fe_zero<P>(); }
  __syncthreads();
  for (uint32_t dd = 1; dd < KATE_THREADS; dd <<= 1) {
    Fe<P> mine = sh[cur][tid];
    if (tid + dd < KATE_THREADS) mine = fe_add(mine, fe_mul(Bp, sh[cur][tid + dd]));
    sh[cur ^ 1][tid] = mine;
    Bp = fe_sqr(Bp);
    cur ^= 1;
    __syncthreads();
  }
  if (totals_out) {                                             // r[s_lo] under a zero carry-in
    if (tid == 0) fe_store(totals_out + slot, sh[cur][0]);
    return;
  }
  // carry-in for this thread = r[hi] = (zero-carry scan value of the next thread) + pt^(s_hi - hi) * (slice carry-in)
  Fe<P> carry = (tid + 1 < KATE_THREADS) ? sh[cur][tid + 1] : fe_zero<P>();
  if (carry_in && lo < hi) carry = fe_add(carry, fe_mul(fe_pow_u64<P>(pt, s_hi - hi), fe_load(carry_in + slot)));
  r = carry;
  for (uint32_t i = hi; i > lo; --i) {
    Fe<P> ai = (i < n) ? fe_load(a + i) : fe_zero<P>();
    r = fe_add(ai, fe_mul(pt, r));
    fe_store(q + i - 1, r);
  }
}
// carries[z] = r[slice_hi(z)], chained from the top slice down: one thread per (division, proof)
template <class P>
__global__ void kate_carry_kernel(uint32_t n, uint32_t splits, uint32_t ndiv, uint32_t batch, const KateDesc* __restrict__ descs,
                                  const Fe<P>* __restrict__ consts, uint32_t cstride, const Fe<P>* __restrict__ totals, Fe<P>* __restrict__ carries) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ndiv * batch) return;
  const uint32_t b = t / ndiv, di = t % ndiv;
  const Fe<P> pt = fe_load(consts + (uint64_t)b * cstride + descs[di].point_const);
  const uint32_t slice = (n + splits - 1) / splits;
  const uint64_t base = ((uint64_t)b * ndiv + di) * splits;
  Fe<P> top = fe_zero<P>();
  for (int z = (int)splits - 1; z >= 0; --z) {
    const uint32_t s_lo = min((uint32_t)z * slice, n), s_hi = min(s_lo + slice, n);
    fe_store(carries + base + z, top);
    top = fe_add(fe_load(totals + base + z), fe_mul(fe_pow_u64<P>(pt, s_hi - s_lo), top));
  }
}

// ---- element tweaks: dst[b][index] = (op 0: dst - v) (op 1: v) where v = vals[b*vstride + vidx] ---------------
template <class P>
__global__ void tweak_element_kernel(Regions reg, uint64_t len, PolyRef dst, uint32_t index, const Fe<P>* __restrict__ vals,
                                     uint32_t vstride, uint32_t vidx, int op, uint32_t batch) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  Fe<P>* p = region_ptr<P>(reg, dst, b, len) + index;
  Fe<P> v = fe_load(vals + (uint64_t)b * vstride + vidx);
  fe_store(p, op == 0 ? fe_sub(fe_load(p), v) : v);
}

// out[b][i] = first * base^i  (b-vector of the IPA, omega powers)
template <class P>
__global__ void powers_kernel(Regions reg, uint32_t n, PolyRef out, const Fe<P>* __restrict__ consts, uint32_t cstride, uint32_t base_const) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b = blockIdx.y;
  if (i >= n) return;
  Fe<P> x = fe_load(consts + (uint64_t)b * cstride + base_const);
  fe_store(region_ptr<P>(reg, out, b, n) + i, fe_pow_u64<P>(x, i));
}

// ---- IPA round kernels ---------------------------------------------------------------------------------
// scalars over the ORIGINAL generators g[0..n):  o = i' + t*(2*half);  G'_j[i'] = sum_t coef[o] g[o]
//   L_j uses p'[half + i'] on i' <  half,   R_j uses p'[i' - half] on i' >= half
template <class P>
// `count` = length of the generator vector the scalars refer to: n, or the length of the materialised G' (prover.cu step 21)
__global__ void ipa_scalars_kernel(Regions reg, uint32_t n, uint32_t count, uint32_t half, PolyRef pprime, PolyRef coef, PolyRef scl, PolyRef scr) {
  uint32_t o = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b = blockIdx.y;
  if (o >= count) return;
  uint32_t ip = o & (2 * half - 1);
  const Fe<P>* pp = region_ptr<P>(reg, pprime, b, n);
  Fe<P> c = fe_load(region_ptr<P>(reg, coef, b, n) + o);
  Fe<P> v = fe_mul(c, fe_load(pp + (ip ^ half)));
  Fe<P> z = fe_zero<P>();
  fe_store(region_ptr<P>(reg, scl, b, n) + o, ip < half ? v : z);
  fe_store(region_ptr<P>(reg, scr, b, n) + o, ip < half ? z : v);
}

// value_l = <p'[half..2half], b[0..half]>, value_r = <p'[0..half], b[half..2half]>; writes the MSM "extra"
// scalars  extraL = [l_rand, value_l * z], extraR = [r_rand, value_r * z]   (points w, u of the g-basis table)
constexpr int IPA_THREADS = 256;
template <class P>
__global__ void __launch_bounds__(IPA_THREADS) ipa_inner_kernel(Regions reg, uint32_t n, uint32_t half, PolyRef pprime, PolyRef bvec,
                                 const Fe<P>* __restrict__ consts, uint32_t cstride, uint32_t z_const,
                                 const Fe<P>* __restrict__ rnd, uint64_t rnd_stride, uint32_t l_rand_idx, uint32_t r_rand_idx,
                                 Fe<P>* __restrict__ extra /* [b][2][2] */) {
  __shared__ Fe<P> shl[IPA_THREADS], shr[IPA_THREADS];
  const uint32_t b = blockIdx.x, tid = threadIdx.x;
  const Fe<P>* pp = region_ptr<P>(reg, pprime, b, n);
  const Fe<P>* bv = region_ptr<P>(reg, bvec, b, n);
  Fe<P> al = fe_zero<P>(), ar = fe_zero<P>();
  for (uint32_t i = tid; i < half; i += IPA_THREADS) {
    al = fe_add(al, fe_mul(fe_load(pp + half + i), fe_load(bv + i)));
    ar = fe_add(ar, fe_mul(fe_load(pp + i), fe_load(bv + half + i)));
  }
  shl[tid] = al; shr[tid] = ar;
  __syncthreads();
  for (uint32_t d = IPA_THREADS >> 1; d > 0; d >>= 1) {
    if (tid < d) { shl[tid] = fe_add(shl[tid], shl[tid + d]); shr[tid] = fe_add(shr[tid], shr[tid + d]); }
    __syncthreads();
  }
  if (tid == 0) {
    Fe<P> z = fe_load(consts + (uint64_t)b * cstride + z_const);
    Fe<P>* e = extra + (uint64_t)b * 4;
    fe_store(e + 0, fe_load(rnd + (uint64_t)b * rnd_stride + l_rand_idx));
    fe_store(e + 1, fe_mul(shl[0], z));
    fe_store(e + 2, fe_load(rnd + (uint64_t)b * rnd_stride + r_rand_idx));
    fe_store(e + 3, fe_mul(shr[0], z));
  }
}

// The same two inner products for a LONG vector (one large proof: half up to 2^19): grid = (proofs, parts), every CTA sums a
// slice into tmp[b][part][2]; ipa_inner_finish_kernel (parts threads per proof) adds the slices and writes the extras.
template <class P>
__global__ void __launch_bounds__(IPA_THREADS) ipa_inner_partial_kernel(Regions reg, uint32_t n, uint32_t half, PolyRef pprime, PolyRef bvec, Fe<P>* __restrict__ tmp) {
  __shared__ Fe<P> shl[IPA_THREADS], shr[IPA_THREADS];
  const uint32_t b = blockIdx.x, part = blockIdx.y, parts = gridDim.y, tid = threadIdx.x;
  const Fe<P>* pp = region_ptr<P>(reg, pprime, b, n);
  const Fe<P>* bv = region_ptr<P>(reg, bvec, b, n);
  const uint32_t per = (half + parts - 1) / parts, lo = part * per, hi = min(half, lo + per);
  Fe<P> al = fe_zero<P>(), ar = fe_zero<P>();
  for (uint32_t i = lo + tid; i < hi; i += IPA_THREADS) {
    al = fe_add(al, fe_mul(fe_load(pp + half + i), fe_load(bv + i)));
    ar = fe_add(ar, fe_mul(fe_load(pp + i), fe_load(bv + half + i)));
  }
  shl[tid] = al; shr[tid] = ar;
  __syncthreads();
  for (uint32_t d = IPA_THREADS >> 1; d > 0; d >>= 1) {
    if (tid < d) { shl[tid] = fe_add(shl[tid], shl[tid + d]); shr[tid] = fe_add(shr[tid], shr[tid + d]); }
    __syncthreads();
  }
  if (tid == 0) { fe_store(tmp + ((uint64_t)b * parts + part) * 2, shl[0]); fe_store(tmp + ((uint64_t)b * parts + part) * 2 + 1, shr[0]); }
}
template <class P>
__global__ void __launch_bounds__(128) ipa_inner_finish_kernel(const Fe<P>* __restrict__ tmp, uint32_t parts,
                                 const Fe<P>* __restrict__ consts, uint32_t cstride, uint32_t z_const,
                                 const Fe<P>* __restrict__ rnd, uint64_t rnd_stride, uint32_t l_rand_idx, uint32_t r_rand_idx, Fe<P>* __restrict__ extra) {
  __shared__ Fe<P> shl[128], shr[128];
  const uint32_t b = blockIdx.x, tid = threadIdx.x;
  shl[tid] = tid < parts ? fe_load(tmp + ((uint64_t)b * parts + tid) * 2) : fe_zero<P>();
  shr[tid] = tid < parts ? fe_load(tmp + ((uint64_t)b * parts + tid) * 2 + 1) : fe_zero<P>();
  __syncthreads();
  for (uint32_t d = 64; d > 0; d >>= 1) {
    if (tid < d) { shl[tid] = fe_add(shl[tid], shl[tid + d]); shr[tid] = fe_add(shr[tid], shr[tid + d]); }
    __syncthreads();
  }
  if (tid == 0) {
    Fe<P> z = fe_load(consts + (uint64_t)b * cstride + z_const);
    Fe<P>* e = extra + (uint64_t)b * 4;
    fe_store(e + 0, fe_load(rnd + (uint64_t)b * rnd_stride + l_rand_idx));
    fe_store(e + 1, fe_mul(shl[0], z));
    fe_store(e + 2, fe_load(rnd + (uint64_t)b * rnd_stride + r_rand_idx));
    fe_store(e + 3, fe_mul(shr[0], z));
  }
}

// p'[i] += u^-1 p'[i+half];  b[i] += u b[i+half]  (i < half);  coef[o] *= u where bit (o / half) is odd
template <class P>
__global__ void ipa_fold_kernel(Regions reg, uint32_t n, uint32_t count, uint32_t half, PolyRef pprime, PolyRef bvec, PolyRef coef,
                                const Fe<P>* __restrict__ consts, uint32_t cstride, uint32_t u_const, uint32_t uinv_const) {
  uint32_t o = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b = blockIdx.y;
  if (o >= count) return;
  const Fe<P>* cb = consts + (uint64_t)b * cstride;
  Fe<P> u = fe_load(cb + u_const);
  if ((o / half) & 1) {
    Fe<P>* c = region_ptr<P>(reg, coef, b, n) + o;
    fe_store(c, fe_mul(fe_load(c), u));
  }
  if (o < half) {
    Fe<P> uinv = fe_load(cb + uinv_const);
    Fe<P>* pp = region_ptr<P>(reg, pprime, b, n);
    Fe<P>* bv = region_ptr<P>(reg, bvec, b, n);
    fe_store(pp + o, fe_add(fe_load(pp + o), fe_mul(uinv, fe_load(pp + o + half))));
    fe_store(bv + o, fe_add(fe_load(bv + o), fe_mul(u, fe_load(bv + o + half))));
  }
}

// fill an array with a constant (coef := 1, instance padding := 0)
template <class P>
__global__ void fill_kernel(Regions reg, uint64_t len, PolyRef dst, uint32_t count, Fe<P> v) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t b = blockIdx.y;
  if (i >= count) return;
  fe_store(region_ptr<P>(reg, dst, b, len) + i, v);
}

}  // namespace bz
