// create_proof on the device, batch-major (B independent proofs in lockstep).
// Mirrors halo2_proofs 0.2.0 `plonk::create_proof` and the argument provers it drives
// (U: src/plonk/prover.rs, src/plonk/{permutation,lookup,vanishing}/prover.rs, src/poly/multiopen/prover.rs,
//  src/poly/commitment/prover.rs, src/transcript.rs; protocol order = SURVEY App. A steps 0-21).
// Host work here is exactly what stays in Rust in the drop-in: Blake2b transcript, challenge bookkeeping,
// blind arithmetic, the lookup sort/permute and multiopen set bookkeeping.  Everything that touches an n- or
// 8n-sized array runs in the kernels of ntt.cu / fixedmsm.cu / poly.cuh.
#include "prover_impl.h"

namespace bz {

// ------------------------------------------------------------------------------------------------------
template <class P> __global__ void geometric_kernel(::bz::Fe<P>* out, ::bz::Fe<P> first, ::bz::Fe<P> base, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  fe_store(out + i, fe_mul(first, fe_pow_u64<P>(base, i)));
}

static DFe dfe(const HFe& h) { DFe r; memcpy(r.l, h.l, 32); return r; }

// pk.permutation.permutations from the copy-constraint cycles (U: plonk/permutation/keygen.rs `Assembly::build_pk`):
// sigma_j[i] = delta^{col'} * omega^{row'}  where (col', row') = mapping[j][i]
template <class P> __global__ void sigma_from_mapping_kernel(const uint32_t* __restrict__ mapping, const ::bz::Fe<P>* __restrict__ omega_pows,
                                                             const ::bz::Fe<P>* __restrict__ delta_pows, ::bz::Fe<P>* __restrict__ out, uint64_t total) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const uint32_t c = mapping[2 * i], r = mapping[2 * i + 1];
  fe_store(out + i, fe_mul(fe_load(delta_pows + c), fe_load(omega_pows + r)));
}

// emit one expression (postfix tokens [lo,hi)); advice -> per-proof slot col, instance -> slot G + col, fixed -> shared slot col
static void emit_tokens(ProgBuilder& pb, const CircuitCopy& cs, const std::vector<Token>& tokens, uint32_t lo, uint32_t hi) {
  for (uint32_t t = lo; t < hi; ++t) {
    const Token& k = tokens[t];
    switch (k.op) {
      case 0: pb.pc(k.a); break;
      case 1: pb.pp(k.a, k.b); break;
      case 2: pb.ps(k.a, k.b); break;
      case 3: pb.pp(cs.G + k.a, k.b); break;
      case 4: pb.neg(); break;
      case 5: pb.add(); break;
      case 6: pb.mul(); break;
      case 7: pb.mulc(k.a); break;
      default: throw Error(-1, "bad token op");
    }
  }
}
static void emit_expr(ProgBuilder& pb, const CircuitCopy& cs, uint32_t lo, uint32_t hi) { emit_tokens(pb, cs, cs.tokens, lo, hi); }

static void derive_fixed_subexpressions(PkImpl& pk) {
  split_fixed_subexpressions(pk.cs.tokens, pk.cs.gate_off, pk.cs.F + pk.M + 5, pk.derived, pk.qtokens, pk.qgate_off);
}

static void emit_compressed(ProgBuilder& pb, const CircuitCopy& cs, const std::vector<std::pair<uint32_t, uint32_t>>& exprs, uint32_t c_theta) {
  for (size_t e = 0; e < exprs.size(); ++e) {
    if (e > 0) pb.mulc(c_theta);
    emit_expr(pb, cs, exprs[e].first, exprs[e].second);
    if (e > 0) pb.add();
  }
}

static uint32_t shslot_fixed(const PkImpl& pk, uint32_t c) { return c; }
static uint32_t shslot_sigma(const PkImpl& pk, uint32_t j) { return pk.cs.F + j; }
static uint32_t shslot_l0(const PkImpl& pk) { return pk.cs.F + pk.M; }
static uint32_t shslot_llast(const PkImpl& pk) { return pk.cs.F + pk.M + 2; }
static uint32_t shslot_active(const PkImpl& pk) { return pk.cs.F + pk.M + 3; }
static uint32_t shslot_x(const PkImpl& pk) { return pk.cs.F + pk.M + 4; }

static void push_column(ProgBuilder& pb, const PkImpl& pk, std::pair<uint32_t, uint32_t> col) {
  if (col.first == 0) pb.pp(col.second, 0);
  else if (col.first == 1) pb.ps(shslot_fixed(pk, col.second), 0);
  else pb.pp(pk.slot_inst(col.second), 0);
}

static void build_programs(PkImpl& pk) {
  const CircuitCopy& cs = pk.cs;
  // ---- lookup compression on the Lagrange domain: outputs 2l (input), 2l+1 (table)
  {
    ProgBuilder pb; pb.scale = 1;
    for (uint32_t l = 0; l < pk.L; ++l) {
      emit_compressed(pb, cs, cs.lookups[l].inputs, pk.C_THETA); pb.store(2 * l);
      emit_compressed(pb, cs, cs.lookups[l].tables, pk.C_THETA); pb.store(2 * l + 1);
    }
    BZ_CHECK(pb.max_depth <= EVAL_STACK, "lookup expression too deep for the evaluator stack");
    pk.lk_ninstr = (uint32_t)pb.code.size();
    if (pb.rot_table.empty()) pb.rot_table.push_back(0);
    pk.h_lk_code = pb.code; pk.h_lk_rot = pb.rot_table;
  }
  // ---- h(X) on the extended coset (SURVEY App. A step 11):  N(X) = sum_e y^(E-1-e) expr_e(X),  h = N / t.
  // Every expr_e of a satisfying witness vanishes on the whole domain, so it is divisible by t(X) = X^n - 1 on its own and
  // expr_e / t has degree < (deg_e - 1) n.  Terms with (deg_e - 1) n <= ext_n / 2 are therefore evaluated on every SECOND
  // point of the extended coset only (that is the coset of the half-size domain), interpolated by a half-size inverse NTT
  // and added to the rest in coefficient form: same h(X), about a third fewer field multiplications for Shot / Board.
  // (For a witness that violates a gate this is not a polynomial identity: the proof differs from that of a single full-coset
  // evaluation, and both are rejected.)
  {
    struct Term { uint32_t degree; std::function<void(ProgBuilder&)> emit; bool gate = false; uint32_t lo = 0, hi = 0; };
    std::vector<Term> terms;
    const uint32_t derived_base = cs.F + pk.M + 5;
    auto degree_of = [&](const std::vector<Token>& tokens, uint32_t lo, uint32_t hi) {
      std::vector<uint32_t> st;
      for (uint32_t t = lo; t < hi; ++t) {
        const Token& k = tokens[t];
        switch (k.op) {
          case 0: st.push_back(0); break;
          case 2: st.push_back(k.a >= derived_base ? pk.derived[k.a - derived_base].degree : 1u); break;
          case 1: case 3: st.push_back(1); break;
          case 4: case 7: break;
          case 5: { uint32_t r = st.back(); st.pop_back(); st.back() = std::max(st.back(), r); break; }
          case 6: { uint32_t r = st.back(); st.pop_back(); st.back() += r; break; }
          default: throw Error(-1, "bad token op");
        }
      }
      return st.back();
    };
    auto expr_degree = [&](uint32_t lo, uint32_t hi) { return degree_of(cs.tokens, lo, hi); };
    auto compressed_degree = [&](const std::vector<std::pair<uint32_t, uint32_t>>& es) { uint32_t d = 0; for (auto& r : es) d = std::max(d, expr_degree(r.first, r.second)); return d; };
    const int last_rot = -((int)cs.bf + 1);
    for (size_t g = 0; g + 1 < pk.qgate_off.size(); ++g) {
      const uint32_t lo = pk.qgate_off[g], hi = pk.qgate_off[g + 1];
      BZ_CHECK(degree_of(pk.qtokens, lo, hi) == expr_degree(cs.gate_off[g], cs.gate_off[g + 1]), "internal: derived columns changed a gate's degree");
      terms.push_back({degree_of(pk.qtokens, lo, hi), [&cs, &pk, lo, hi](ProgBuilder& pb) { emit_tokens(pb, cs, pk.qtokens, lo, hi); }, true, lo, hi});
    }
    if (pk.nsets) {
      terms.push_back({2, [&pk](ProgBuilder& pb) { pb.pc(pk.C_ONE); pb.pp(pk.slot_pz(0), 0); pb.sub(); pb.ps(shslot_l0(pk), 0); pb.mul(); }});          // l0 * (1 - z_0)
      terms.push_back({3, [&pk](ProgBuilder& pb) { uint32_t zl = pk.slot_pz(pk.nsets - 1);                                                               // l_last * (z_l^2 - z_l)
                                                   pb.pp(zl, 0); pb.pp(zl, 0); pb.mul(); pb.pp(zl, 0); pb.sub(); pb.ps(shslot_llast(pk), 0); pb.mul(); }});
      for (uint32_t i = 1; i < pk.nsets; ++i)                                                                                                            // l0 * (z_i - z_{i-1}(w^last X))
        terms.push_back({2, [&pk, i, last_rot](ProgBuilder& pb) { pb.pp(pk.slot_pz(i), 0); pb.pp(pk.slot_pz(i - 1), last_rot); pb.sub(); pb.ps(shslot_l0(pk), 0); pb.mul(); }});
      for (uint32_t s = 0; s < pk.nsets; ++s) {
        const uint32_t c0 = s * pk.chunk_len, c1 = std::min<uint32_t>(pk.M, c0 + pk.chunk_len);
        terms.push_back({c1 - c0 + 2, [&pk, &cs, s, c0, c1](ProgBuilder& pb) {
          pb.pp(pk.slot_pz(s), 1);
          for (uint32_t j = c0; j < c1; ++j) { push_column(pb, pk, cs.perm[j]); pb.ps(shslot_sigma(pk, j), 0); pb.mulc(pk.C_BETA); pb.add(); pb.addc(pk.C_GAMMA); pb.mul(); }
          pb.pp(pk.slot_pz(s), 0);
          for (uint32_t j = c0; j < c1; ++j) { push_column(pb, pk, cs.perm[j]); pb.ps(shslot_x(pk), 0); pb.mulc(pk.C_BD0 + j); pb.add(); pb.addc(pk.C_GAMMA); pb.mul(); }
          pb.sub(); pb.ps(shslot_active(pk), 0); pb.mul(); }});
      }
    }
    for (uint32_t l = 0; l < pk.L; ++l) {
      const uint32_t a = pk.slot_lk(l, 0), sp = pk.slot_lk(l, 1), z = pk.slot_lk(l, 2);
      terms.push_back({2, [&pk, z](ProgBuilder& pb) { pb.pc(pk.C_ONE); pb.pp(z, 0); pb.sub(); pb.ps(shslot_l0(pk), 0); pb.mul(); }});
      terms.push_back({3, [&pk, z](ProgBuilder& pb) { pb.pp(z, 0); pb.pp(z, 0); pb.mul(); pb.pp(z, 0); pb.sub(); pb.ps(shslot_llast(pk), 0); pb.mul(); }});
      // z(wX)(a'+beta)(s'+gamma) - z(X)(A_theta+beta)(S_theta+gamma)
      const uint32_t dprod = std::max(3u, 1 + compressed_degree(cs.lookups[l].inputs) + compressed_degree(cs.lookups[l].tables)) + 1;
      terms.push_back({dprod, [&pk, &cs, l, a, sp, z](ProgBuilder& pb) {
        pb.pp(z, 1); pb.pp(a, 0); pb.addc(pk.C_BETA); pb.mul(); pb.pp(sp, 0); pb.addc(pk.C_GAMMA); pb.mul();
        pb.pp(z, 0);
        emit_compressed(pb, cs, cs.lookups[l].inputs, pk.C_THETA); pb.addc(pk.C_BETA); pb.mul();
        emit_compressed(pb, cs, cs.lookups[l].tables, pk.C_THETA); pb.addc(pk.C_GAMMA); pb.mul();
        pb.sub(); pb.ps(shslot_active(pk), 0); pb.mul(); }});
      terms.push_back({2, [&pk, a, sp](ProgBuilder& pb) { pb.pp(a, 0); pb.pp(sp, 0); pb.sub(); pb.ps(shslot_l0(pk), 0); pb.mul(); }});                     // l0 * (a' - s')
      terms.push_back({3, [&pk, a, sp](ProgBuilder& pb) { pb.pp(a, 0); pb.pp(sp, 0); pb.sub(); pb.pp(a, 0); pb.pp(a, -1); pb.sub(); pb.mul(); pb.ps(shslot_active(pk), 0); pb.mul(); }});
    }
    BZ_CHECK(terms.size() == pk.n_exprs, "internal: expression count mismatch");
    const bool tiers = pk.ext_k > cs.k;
    // tier of a term: the largest t <= 2 with (deg - 1) n <= ext_n >> t  (and at least n points)
    auto tier_of = [&](uint32_t degree) {
      uint32_t t = 0;
      if (!tiers) return t;
      while (t + 1 < PkImpl::Q_TIERS && (pk.ext_n >> (t + 1)) >= pk.n && (uint64_t)(degree - 1) * pk.n <= (pk.ext_n >> (t + 1))) ++t;
      return t;
    };
    // BZ_QUOTIENT_CSE=0: every gate polynomial as its own expression tree (the reference's evaluation order), for A/B runs
    const char* cse_env = getenv("BZ_QUOTIENT_CSE");
    const bool use_dag = !(cse_env && atoi(cse_env) == 0);
    auto count_muls = [](const ProgBuilder& pb) {
      uint32_t m = 0;
      for (uint32_t ins : pb.code) { const uint32_t op = ins & 15u; m += op == OP_MUL || op == OP_MULC || op == OP_FOLD || op == OP_ACC_MULC || op == OP_MUL_T_STORE; }
      return m;
    };
    // one tier's program; variant 0: direct common factors only, 1: through nested products too, 2: products as sorted chains
    // of their factors as well (evalprog.h)
    auto compile = [&](uint32_t tier, int variant, ProgBuilder& pb) {
      pb.scale = 1 << (pk.ext_k - cs.k);
      const uint32_t E = (uint32_t)terms.size();
      auto yp = [&pk](uint32_t d) { return pk.C_YP0 + d; };
      int prev = -1;
      // the gate polynomials of this tier: one DAG (shared sub-expressions once, common factors hoisted; evalprog.h)
      GateDag dag; dag.advice_slot_of_instance = cs.G; dag.nested = variant >= 1; dag.canon_mul = dag.sort_rest = variant >= 2;
      if (use_dag) {
        for (uint32_t e = 0; e < E; ++e)
          if (terms[e].gate && tier_of(std::max(1u, terms[e].degree)) == tier) dag.add(pk.qtokens, terms[e].lo, terms[e].hi, e);
        dag.plan();
        for (const GateDag::Group& g : dag.groups) {
          dag.emit_group(pb, g, prev, yp);
          prev = (int)dag.polys[g.first + g.count - 1].e;
        }
      }
      for (uint32_t e = 0; e < E; ++e) {
        if ((use_dag && terms[e].gate) || tier_of(std::max(1u, terms[e].degree)) != tier) continue;
        terms[e].emit(pb);
        pb.fold(yp(prev < 0 ? 1u : e - (uint32_t)prev));          // acc = acc * y^(gap) + expr
        prev = (int)e;
      }
      if (prev < 0) return false;                                            // nothing in this tier
      if ((uint32_t)prev != E - 1) pb.accmul(pk.C_YP0 + (E - 1 - (uint32_t)prev));
      pb.code.push_back(OP_MUL_T_STORE);
      return true;
    };
    auto build = [&](uint32_t tier, uint32_t& ninstr) {
      ProgBuilder pb;
      ninstr = 0; pk.q_muls[tier] = 0; pk.h_q_code[tier].clear(); pk.h_q_rot[tier].clear();
      if (!compile(tier, 0, pb)) return;
      for (int variant = 1; use_dag && variant <= 2; ++variant) {            // re-association can win or lose sharing: keep the cheapest program
        ProgBuilder alt;
        compile(tier, variant, alt);
        if (alt.max_depth <= EVAL_STACK && (pb.max_depth > EVAL_STACK || count_muls(alt) < count_muls(pb))) pb = alt;
      }
      BZ_CHECK(pb.max_depth <= EVAL_STACK, "gate expression too deep for the evaluator stack");
      ninstr = (uint32_t)pb.code.size();
      pk.q_muls[tier] = count_muls(pb);
      BZ_CHECK(ninstr * 4 <= 96 * 1024, "quotient program too large for shared memory");
      if (pb.rot_table.empty()) pb.rot_table.push_back(0);
      pk.h_q_code[tier] = pb.code; pk.h_q_rot[tier] = pb.rot_table;
    };
    for (uint32_t t = 0; t < PkImpl::Q_TIERS; ++t) build(t, pk.q_ninstr[t]);
    BZ_CHECK(pk.q_ninstr[0] > 0, "internal: no full-degree term in h(X)");
  }
}

// programs -> device; the circuit-specialised straight-line kernel of a tier is looked up by the hash of its program
static void upload_programs(PkImpl& pk) {
  auto up = [](DevBuf& d, const void* src, size_t bytes) { if (bytes) { d.alloc(bytes); BZ_CUDA(cudaMemcpy(d.p, src, bytes, cudaMemcpyHostToDevice)); } };
  up(pk.lk_code, pk.h_lk_code.data(), pk.h_lk_code.size() * 4);
  up(pk.lk_rot, pk.h_lk_rot.data(), pk.h_lk_rot.size() * 4);
  const char* env = getenv("BZ_QUOTIENT_GENERATED");            // =0: always the interpreter (A/B)
  const bool use_gen = !(env && atoi(env) == 0);
  for (uint32_t t = 0; t < PkImpl::Q_TIERS; ++t) {
    up(pk.q_code[t], pk.h_q_code[t].data(), pk.h_q_code[t].size() * 4);
    up(pk.q_rot[t], pk.h_q_rot[t].data(), pk.h_q_rot[t].size() * 4);
    pk.q_gen[t] = use_gen && pk.q_ninstr[t] ? find_generated_quotient(program_hash(pk.h_q_code[t], pk.h_q_rot[t])) : nullptr;
  }
}

// ------------------------------------------------------------------------------------------------------
static void add_query(VkImpl& pk, int cid, int rot, PolyRef poly, int bk, int bi, int ev = -1) { pk.queries.push_back(Query{cid, rot, poly, bk, bi, ev}); }

// static structure of the multiopen argument (U: multiopen.rs::construct_intermediate_sets); points are
// identified by their rotation (x * omega^rot are distinct for distinct rotations)
static void build_multiopen(VkImpl& pk) {
  std::vector<int> point_order;                       // rotation -> point index = position
  auto point_index = [&](int rot) { for (size_t i = 0; i < point_order.size(); ++i) if (point_order[i] == rot) return (int)i; point_order.push_back(rot); return (int)point_order.size() - 1; };
  struct Tmp { int cid; PolyRef poly; int bk, bi; std::vector<int> pidx; };
  std::vector<Tmp> cm;
  for (const Query& q : pk.queries) {
    int pi = point_index(q.rot);
    auto it = std::find_if(cm.begin(), cm.end(), [&](const Tmp& t) { return t.cid == q.cid; });
    if (it == cm.end()) cm.push_back(Tmp{q.cid, q.poly, q.blind_kind, q.blind_idx, {pi}});
    else it->pidx.push_back(pi);
  }
  std::vector<std::vector<int>> sets;                 // sorted unique point-index sets, first-appearance order
  for (Tmp& t : cm) {
    std::vector<int> s = t.pidx; std::sort(s.begin(), s.end()); s.erase(std::unique(s.begin(), s.end()), s.end());
    int idx = -1;
    for (size_t i = 0; i < sets.size(); ++i) if (sets[i] == s) idx = (int)i;
    if (idx < 0) { sets.push_back(s); idx = (int)sets.size() - 1; }
    pk.cmap.push_back(VkImpl::CommInfo{t.poly, t.bk, t.bi, idx, t.cid});
  }
  for (auto& s : sets) { std::vector<int> r; for (int pi : s) r.push_back(point_order[pi]); pk.point_sets.push_back(r); }
}

// ------------------------------------------------------------------------------------------------------
static void ensure_work(Ctx* ctx, PkImpl& pk, uint32_t B) {
  PkImpl::Work& w = pk.work;
  if (w.batch >= B) return;
  const size_t n = pk.n, en = pk.ext_n, E = 32;
  w.val.alloc(B * pk.NS * n * E);
  w.poly.alloc(B * pk.NS * n * E);
  w.coset.alloc(B * pk.NS * en * E);
  w.misc.alloc(B * pk.NM * n * E);
  w.rnd.alloc(B * (size_t)pk.R * E);
  w.wide.alloc(B * (size_t)pk.R * 64);
  w.hext.alloc(B * en * E);
  w.hcoef.alloc(B * en * E);
  w.hext_low.alloc(B * (en / 2 + en / 4) * E);        // tiers 1 and 2, back to back
  w.hcoef_low.alloc(B * (en / 2) * E);
  w.nd.alloc(4 * (size_t)std::max<uint32_t>(1, pk.nsets + pk.L) * B * n * E);       // num, den, prefix(num), suffix(den) of every grand product
  w.consts.alloc(B * (size_t)pk.cstride * E);
  // commitment requests per proof in one call: advice columns, 2 per lookup, grand products, the h pieces (or 2 IPA terms)
  const size_t max_req = std::max<size_t>((size_t)pk.cs.G + pk.cs.I, std::max<size_t>(std::max<size_t>(2 * pk.L, pk.nsets + pk.L), std::max<size_t>(pk.qdeg, 2)));
  w.extras.alloc(B * max_req * 2 * E);
  w.evalout.alloc(B * (pk.evals.size() + pk.point_sets.size() + 8) * E);
  w.commits.alloc(B * max_req * 128);
  w.ptrs.alloc(B * max_req * 2 * sizeof(void*));
  w.descs.alloc(64 * 1024);
  w.lk_sorted.alloc(std::max<size_t>(1, (size_t)B * pk.L * n * E));
  w.lk_err.alloc((size_t)B * 4 + 64);
  if (w.h_err) cudaFreeHost(w.h_err);
  BZ_CUDA(cudaMallocHost(&w.h_err, (size_t)B * 4 + 64));
  if (w.h_pinned) cudaFreeHost(w.h_pinned);
  w.h_pinned_bytes = std::max<size_t>(B * std::max<size_t>(2 * n * E * std::max<uint32_t>(1, pk.L), std::max<size_t>(max_req * 128, (pk.evals.size() + 16) * E)), 1 << 20);
  BZ_CUDA(cudaMallocHost(&w.h_pinned, w.h_pinned_bytes));
  w.batch = B;
}

void params_commit_run(Ctx* C, const ParamsImpl& p, bool lagrange, const void* const* d_main, const void* const* d_extra,
                       uint32_t n_msm, void* d_out, bool xyzz_out) {
  const FixedBase& fb = lagrange ? p.fb_gl : p.fb_g;
  if (p.use_tables) {
    fixed_msm_run(C, fb, d_main, p.n, d_extra, n_msm, d_out, xyzz_out);
    return;
  }
  // bucket MSM (k >= 20, or forced): the MSMs of the call are sorted, accumulated and reduced as ONE batch
  BZ_CHECK(!xyzz_out, "internal: the bucket MSM returns affine commitments only");
  C->commit_jac.ensure((size_t)n_msm * 96);
  msm_run_batch(C, p.curve, d_main, d_extra, p.n, 0, fb.npts, lagrange ? p.gl_w.p : p.g_w_u.p, n_msm, C->commit_jac.p);
  jac_to_affine_run(C, p.curve, C->commit_jac.p, d_out, n_msm);
}

const void* const* upload_msm_ptrs(Ctx* C, DevBuf& d, const std::vector<void*>& mainp, const std::vector<void*>& extrap) {
  const size_t bytes = mainp.size() * sizeof(void*);
  d.ensure(2 * bytes);
  BZ_CUDA(cudaMemcpyAsync(d.p, mainp.data(), bytes, cudaMemcpyHostToDevice, C->stream));
  BZ_CUDA(cudaMemcpyAsync((char*)d.p + bytes, extrap.data(), bytes, cudaMemcpyHostToDevice, C->stream));
  return (const void* const*)d.p;
}

// ------------------------------------------------------------------------------------------------------
}  // namespace bz

using namespace bz;

extern "C" {

API int bz_params_create(bz_ctx* ctx, uint32_t k, int curve, const void* g, const void* g_lagrange, const void* w, const void* u,
                         int window_bits, bz_params** out) {
  PV_TRY(ctx, {
    BZ_CHECK(out && g && g_lagrange && w && u, "null argument");
    BZ_CHECK(k >= 1 && k <= 24, "k out of range");
    BZ_CHECK(curve == 0 || curve == 1, "bad curve id");
    *out = nullptr;
    std::unique_ptr<bz_params> h(new bz_params());
    ParamsImpl& p = h->p;
    p.k = k; p.n = 1u << k; p.curve = curve;
    const size_t n = p.n;
    p.g_w_u.alloc((n + 2) * 64);
    p.gl_w.alloc((n + 1) * 64);
    BZ_CUDA(cudaMemcpy(p.g_w_u.p, g, n * 64, cudaMemcpyHostToDevice));
    BZ_CUDA(cudaMemcpy((char*)p.g_w_u.p + n * 64, w, 64, cudaMemcpyHostToDevice));
    BZ_CUDA(cudaMemcpy((char*)p.g_w_u.p + (n + 1) * 64, u, 64, cudaMemcpyHostToDevice));
    BZ_CUDA(cudaMemcpy(p.gl_w.p, g_lagrange, n * 64, cudaMemcpyHostToDevice));
    BZ_CUDA(cudaMemcpy((char*)p.gl_w.p + n * 64, w, 64, cudaMemcpyHostToDevice));
    uint32_t c = window_bits > 0 ? (uint32_t)window_bits : 0;
    if (!c) {
      const char* e = getenv("BZ_FIXED_WINDOW");
      c = e ? (uint32_t)atoi(e) : 0;
      if (!c) {   // largest window whose two tables stay under 160 GB of the B200's 191 GB (k = 11: c = 16, 138 GB; k = 12: c = 15, 155 GB;
        // k = 13: c = 13, 85 GB) and under 2^31 entries.  Measured on B200, Shot proofs/s: c = 13 -> 2422, 14 -> 2457, 15 -> 2560
        // (17 instead of ~18.8 additions per scalar: the top window of a 255-bit scalar is almost never occupied at c = 15);
        // with 6 lanes: c = 15 -> 3250, c = 16 -> 3324 (16 additions); Board c = 14 -> 15: table MSM time -9 %.
        // The cap also respects what is free right now, so a second Params alive at the same time gets a smaller window.
        size_t free_b = 0, total_b = 0;
        BZ_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const double cap = std::min(160e9, (double)free_b - 16e9);          // leave room for the batch work areas
        for (c = std::min(16u, std::max(8u, k + 5)); c > 4; --c) {
          double entries = (double)((256 + c - 1) / c) * (double)(1u << (c - 1)) * (double)(n + 2);
          if (2.0 * entries * 64.0 <= cap && entries < 2147483648.0) break;
        }
      }
    }
    const char* fg = getenv("BZ_FORCE_GENERAL_MSM");
    // k <= 19: window tables (k = 18: c = 7, 37 additions per scalar at ~6 G additions/s = 6.2 ns against 13.9 ns per point
    // for the bucket MSM at 2^18; k = 19: c = 6, 7.2 ns against ~9); k >= 20: the bucket MSM wins (6.3 ns at 2^20) and the
    // tables would not fit
    p.use_tables = k <= 19 && !(fg && atoi(fg));
    if (p.use_tables) {
      fixed_base_build(C, p.fb_g, curve, p.g_w_u.p, (uint32_t)n + 2, c);
      fixed_base_build(C, p.fb_gl, curve, p.gl_w.p, (uint32_t)n + 1, c);
    } else {
      p.fb_g.curve = p.fb_gl.curve = curve; p.fb_g.npts = (uint32_t)n + 2; p.fb_gl.npts = (uint32_t)n + 1;
    }
    *out = h.release();
  });
}

API void bz_params_destroy(bz_params* params) { delete params; }

API int bz_params_commit(bz_ctx* ctx, bz_params* params, int lagrange_basis, const void* poly, const void* blind, void* out_affine) {
  PV_TRY(ctx, {
    BZ_CHECK(params && poly && blind && out_affine, "null argument");
    ParamsImpl& p = params->p;
    cudaStream_t st = C->stream;
    DevBuf &d_poly = C->stage[0], &d_out = C->stage[1], &d_extra = C->stage[3], &d_ptrs = C->stage[4];
    d_poly.ensure((size_t)p.n * 32); d_out.ensure(64); d_extra.ensure(64);
    BZ_CUDA(cudaMemcpyAsync(d_poly.p, poly, (size_t)p.n * 32, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaMemsetAsync(d_extra.p, 0, 64, st));
    BZ_CUDA(cudaMemcpyAsync(d_extra.p, blind, 32, cudaMemcpyHostToDevice, st));
    const void* const* d = upload_msm_ptrs(C, d_ptrs, {d_poly.p}, {d_extra.p});
    params_commit_run(C, p, lagrange_basis, d, d + 1, 1, d_out.p);
    BZ_CUDA(cudaMemcpyAsync(out_affine, d_out.p, 64, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}

// Params::commit / commit_lagrange for `count` device-resident polynomials at once (count x n scalars, contiguous;
// blinds: count scalars) -> count affine points on the device.  The unit of work the north star shards across GPUs
// ("independent column commitments ... per GPU"): each rank commits its share of the columns, the 64 B results are
// all-gathered (sharding.py).
API int bz_params_commit_batch_dev(bz_ctx* ctx, bz_params* params, int lagrange_basis, const void* d_polys, const void* d_blinds,
                                   uint32_t count, void* d_out_affine) {
  PV_TRY(ctx, {
    BZ_CHECK(params && d_polys && d_blinds && d_out_affine, "null argument");
    if (!count) return BZ_OK;
    ParamsImpl& p = params->p;
    cudaStream_t st = C->stream;
    const FixedBase& fb = lagrange_basis ? p.fb_gl : p.fb_g;
    const uint32_t nextra = fb.npts - p.n;
    // persistent staging (no cudaMalloc / cudaFree per call: large frees stall the whole device for 100+ ms now and then)
    DevBuf &d_extra = C->stage[3], &d_ptrs = C->stage[4];
    d_extra.ensure((size_t)count * nextra * 32);
    BZ_CUDA(cudaMemsetAsync(d_extra.p, 0, (size_t)count * nextra * 32, st));
    BZ_CUDA(cudaMemcpy2DAsync(d_extra.p, (size_t)nextra * 32, d_blinds, 32, 32, count, cudaMemcpyDeviceToDevice, st));   // blind -> the w slot
    std::vector<void*> mainp(count), extrap(count);
    for (uint32_t j = 0; j < count; ++j) { mainp[j] = (char*)d_polys + (size_t)j * p.n * 32; extrap[j] = (char*)d_extra.p + (size_t)j * nextra * 32; }
    const void* const* d = upload_msm_ptrs(C, d_ptrs, mainp, extrap);
    params_commit_run(C, p, lagrange_basis, d, d + count, count, d_out_affine);
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}

API void bz_pk_destroy(bz_pk* pk) { delete pk; }
API uint32_t bz_pk_num_random(const bz_pk* pk) { return pk ? pk->p.R : 0; }
API uint32_t bz_pk_proof_size(const bz_pk* pk) { return pk ? pk->p.proof_size : 0; }
API uint32_t bz_pk_quotient_muls(const bz_pk* pk, uint32_t tier, uint32_t* points) {
  if (!pk || tier >= PkImpl::Q_TIERS) return 0;
  if (points) *points = pk->p.q_ninstr[tier] ? pk->p.ext_n >> tier : 0;
  return pk->p.q_muls[tier];
}

}  // extern "C"

namespace bz {

// The verifying key's part of keygen: the flattened constraint system, domain constants, the query list, the multiopen
// structure, the number of evaluations and the proof size.  Needs no GPU.
void vk_host_setup(const bzh::Field& F, VkImpl& vk, const bz_circuit* cin) {
  CircuitCopy& cs = vk.cs;
  cs.k = cin->k; cs.G = cin->num_advice; cs.F = cin->num_fixed; cs.I = cin->num_instance; cs.degree = cin->degree; cs.bf = cin->blinding_factors;
  for (uint32_t i = 0; i < cin->n_advice_queries; ++i) cs.aq.push_back({cin->advice_queries[2 * i], cin->advice_queries[2 * i + 1]});
  for (uint32_t i = 0; i < cin->n_fixed_queries; ++i) cs.fq.push_back({cin->fixed_queries[2 * i], cin->fixed_queries[2 * i + 1]});
  for (uint32_t i = 0; i < cin->n_instance_queries; ++i) cs.iq.push_back({cin->instance_queries[2 * i], cin->instance_queries[2 * i + 1]});
  for (uint32_t i = 0; i < cin->n_perm_columns; ++i) cs.perm.push_back({cin->perm_columns[2 * i], cin->perm_columns[2 * i + 1]});
  cs.consts.resize(cin->n_constants);
  if (cin->n_constants) memcpy(cs.consts.data(), cin->constants, (size_t)cin->n_constants * 32);
  cs.tokens.resize(cin->n_tokens);
  for (uint32_t i = 0; i < cin->n_tokens; ++i) cs.tokens[i] = Token{cin->tokens[i].op, cin->tokens[i].a, cin->tokens[i].b};
  cs.gate_off.assign(cin->gate_poly_offsets, cin->gate_poly_offsets + cin->n_gate_polys + 1);
  {
    uint32_t e = 0;
    for (uint32_t l = 0; l < cin->n_lookups; ++l) {
      CircuitCopy::Lookup lk;
      for (uint32_t j = 0; j < cin->lookup_input_counts[l]; ++j, ++e) lk.inputs.push_back({cin->lookup_expr_offsets[e], cin->lookup_expr_offsets[e + 1]});
      for (uint32_t j = 0; j < cin->lookup_table_counts[l]; ++j, ++e) lk.tables.push_back({cin->lookup_expr_offsets[e], cin->lookup_expr_offsets[e + 1]});
      cs.lookups.push_back(lk);
    }
  }
  {
    uint64_t raw[4]; memcpy(raw, cin->vk_transcript_repr, 32);
    cs.vk_repr = F.from_raw(raw);
  }
  BZ_CHECK(cs.degree >= 3, "cs degree must be >= 3");
  vk.n = 1u << cs.k;
  vk.qdeg = cs.degree - 1;
  vk.M = (uint32_t)cs.perm.size(); vk.L = (uint32_t)cs.lookups.size();
  vk.chunk_len = cs.degree - 2;
  vk.nsets = vk.M ? (vk.M + vk.chunk_len - 1) / vk.chunk_len : 0;
  vk.usable = vk.n - (cs.bf + 1);
  BZ_CHECK(vk.chunk_len <= 8, "permutation chunk too wide");
  // domain constants: omega = ROOT_OF_UNITY^(2^(32-k))
  vk.omega = F.root_of_unity();
  for (uint32_t i = cs.k; i < 32; ++i) vk.omega = F.sqr(vk.omega);
  vk.omega_inv = F.inv(vk.omega);
  // ---- queries (SURVEY App. A step 19).  blind slots: advice[G], lookup (A',S',Z)[3L], perm[nsets], h, random
  auto b_adv = [&](uint32_t g) { return (int)g; };
  auto b_lk = [&](uint32_t l, uint32_t w) { return (int)(cs.G + 3 * l + w); };
  auto b_pz = [&](uint32_t s) { return (int)(cs.G + 3 * vk.L + s); };
  const int b_h = (int)(cs.G + 3 * vk.L + vk.nsets), b_rand = b_h + 1;
  const int last_rot = -((int)cs.bf + 1);
  // positions in the proof's evaluation list (the order pk_host_setup writes it in; steps 14-18)
  const int e_adv0 = (int)cs.iq.size(), e_fix0 = e_adv0 + (int)cs.aq.size(), e_rand = e_fix0 + (int)cs.fq.size(), e_sig0 = e_rand + 1;
  const int e_perm0 = e_sig0 + (int)vk.M;
  auto e_perm = [&](uint32_t s2) { return e_perm0 + 3 * (int)s2; };                     // z, z_next, (z_last: all but the last set)
  const int e_lk0 = e_perm0 + (vk.nsets ? 3 * (int)vk.nsets - 1 : 0);
  for (size_t i = 0; i < cs.iq.size(); ++i) add_query(vk, cid_inst + cs.iq[i].first, cs.iq[i].second, PolyRef{R_POLY, vk.slot_inst(cs.iq[i].first)}, 0, 0, (int)i);
  for (size_t i = 0; i < cs.aq.size(); ++i) add_query(vk, cid_adv + cs.aq[i].first, cs.aq[i].second, PolyRef{R_POLY, (uint32_t)cs.aq[i].first}, 1, b_adv(cs.aq[i].first), e_adv0 + (int)i);
  for (uint32_t s2 = 0; s2 < vk.nsets; ++s2) {
    add_query(vk, cid_pz + s2, 0, PolyRef{R_POLY, vk.slot_pz(s2)}, 1, b_pz(s2), e_perm(s2));
    add_query(vk, cid_pz + s2, 1, PolyRef{R_POLY, vk.slot_pz(s2)}, 1, b_pz(s2), e_perm(s2) + 1);
  }
  for (int s2 = (int)vk.nsets - 2; s2 >= 0; --s2) add_query(vk, cid_pz + s2, last_rot, PolyRef{R_POLY, vk.slot_pz(s2)}, 1, b_pz(s2), e_perm(s2) + 2);
  for (uint32_t l = 0; l < vk.L; ++l) {
    const int e = e_lk0 + 5 * (int)l;                                                   // z, z_next, a, a_inv, s
    add_query(vk, cid_lk + 3 * l + 2, 0, PolyRef{R_POLY, vk.slot_lk(l, 2)}, 1, b_lk(l, 2), e);
    add_query(vk, cid_lk + 3 * l + 0, 0, PolyRef{R_POLY, vk.slot_lk(l, 0)}, 1, b_lk(l, 0), e + 2);
    add_query(vk, cid_lk + 3 * l + 1, 0, PolyRef{R_POLY, vk.slot_lk(l, 1)}, 1, b_lk(l, 1), e + 4);
    add_query(vk, cid_lk + 3 * l + 0, -1, PolyRef{R_POLY, vk.slot_lk(l, 0)}, 1, b_lk(l, 0), e + 3);
    add_query(vk, cid_lk + 3 * l + 2, 1, PolyRef{R_POLY, vk.slot_lk(l, 2)}, 1, b_lk(l, 2), e + 1);
  }
  for (size_t i = 0; i < cs.fq.size(); ++i) add_query(vk, cid_fix + cs.fq[i].first, cs.fq[i].second, PolyRef{R_SHPOLY, (uint32_t)cs.fq[i].first}, 0, 0, e_fix0 + (int)i);
  for (uint32_t j = 0; j < vk.M; ++j) add_query(vk, cid_sig + j, 0, PolyRef{R_SHPOLY, cs.F + j}, 0, 0, e_sig0 + (int)j);
  add_query(vk, cid_h, 0, PolyRef{R_MISC, vk.misc_h()}, 1, b_h, -1);
  add_query(vk, cid_rand, 0, PolyRef{R_RANDPOLY, 0}, 1, b_rand, e_rand);
  build_multiopen(vk);
  vk.nev = (uint32_t)e_lk0 + 5 * vk.L;
  // proof size: points (32 B) + scalars (32 B)
  const uint32_t npoints = cs.G + 2 * vk.L + vk.nsets + vk.L + 1 + vk.qdeg + 1 + 1 + 2 * cs.k;
  const uint32_t nscalars = vk.nev + (uint32_t)vk.point_sets.size() + 2;
  vk.proof_size = 32 * (npoints + nscalars);
}

// Everything of keygen_pk's image that needs no GPU: the verifying key's part (vk_host_setup), then the prover's own layouts of
// the per-proof constants / randomness / polynomial slots, the evaluation list and the compiled programs.
// (Also what bz_quotient_program runs at build time to emit the circuit-specialised kernels.)
static void pk_host_setup(const bzh::Field& F, PkImpl& pk, const bz_circuit* cin) {
  vk_host_setup(F, pk, cin);
  const CircuitCopy& cs = pk.cs;
  pk.ext_k = cs.k;
  while ((1ull << pk.ext_k) < (uint64_t)pk.n * pk.qdeg) ++pk.ext_k;
  pk.ext_n = 1u << pk.ext_k;
  pk.NS = cs.G + cs.I + 3 * pk.L + pk.nsets;
  pk.NC = (uint32_t)cs.consts.size();
  pk.ext_omega = F.root_of_unity();
  for (uint32_t i = pk.ext_k; i < 32; ++i) pk.ext_omega = F.sqr(pk.ext_omega);
  const uint32_t n = pk.n;
  derive_fixed_subexpressions(pk);
  // ---- const table layout
  uint32_t c = pk.NC;
  pk.C_ONE = c++; pk.C_THETA = c++; pk.C_BETA = c++; pk.C_GAMMA = c++; pk.C_Y = c++; pk.C_X = c++; pk.C_XN = c++;
  pk.C_X1 = c++; pk.C_X2 = c++; pk.C_X3 = c++; pk.C_X4 = c++; pk.C_XI = c++; pk.C_Z = c++; pk.C_U = c++; pk.C_UINV = c++;
  pk.C_BD0 = c; c += pk.M;
  {
    std::set<int> rs;
    for (auto& q : cs.aq) rs.insert(q.second);
    for (auto& q : cs.fq) rs.insert(q.second);
    for (auto& q : cs.iq) rs.insert(q.second);
    rs.insert(0); rs.insert(1); rs.insert(-1); rs.insert(-((int)cs.bf + 1));
    pk.C_ROT0 = c;
    for (int r : rs) { pk.rots.push_back(r); pk.rot_const[r] = c++; }
  }
  pk.n_exprs = cin->n_gate_polys + (pk.nsets ? 2 + (pk.nsets - 1) + pk.nsets : 0) + 5 * pk.L;
  pk.C_YP0 = c; c += pk.n_exprs + 1;          // y^0 .. y^E
  pk.cstride = c;
  // ---- randomness layout (SURVEY App. A)
  uint32_t r = 0;
  pk.r_adv_rows = r; r += cs.G * (cs.bf + 1);
  pk.r_adv_blind = r; r += cs.G;
  pk.r_lk0 = r; r += pk.L * (2 * (cs.bf + 1) + 2);
  pk.r_perm0 = r; r += pk.nsets * (cs.bf + 1);
  pk.r_lkz0 = r; r += pk.L * (cs.bf + 1);
  pk.r_randpoly = r; r += n;
  pk.r_rand_blind = r; r += 1;
  pk.r_hblind = r; r += pk.qdeg;
  pk.r_qprime = r; r += 1;
  pk.r_spoly = r; r += n;
  pk.r_sblind = r; r += 1;
  pk.r_ipa = r; r += 2 * cs.k;
  pk.R = r;
  // ---- per-proof blind slots of the queries: advice[G], lookup (A',S',Z)[3L], perm[nsets], h, random
  pk.nblinds = cs.G + 3 * pk.L + pk.nsets + 2;
  // ---- MISC slots
  uint32_t m = 0;
  pk.m_cin0 = m; m += 2 * pk.L;
  pk.m_hpoly = m++;                           // = misc_h(), the slot the h(X) query names
  const uint32_t nps = (uint32_t)pk.point_sets.size();
  pk.m_qset0 = m; m += nps;
  pk.m_qtmp0 = m; m += 2 * nps;
  pk.m_qprime = m++; pk.m_ppoly = m++; pk.m_pprime = m++; pk.m_b = m++; pk.m_coef = m++; pk.m_scl = m++; pk.m_scr = m++;
  pk.NM = m;
  // ---- evaluation list in transcript order (steps 14-18)
  const int last_rot = -((int)cs.bf + 1);
  auto ev = [&](PolyRef p, int rot) { pk.evals.push_back(EvalQuery{p, pk.rot_const.at(rot)}); };
  for (auto& q : cs.iq) ev(PolyRef{R_POLY, pk.slot_inst(q.first)}, q.second);
  for (auto& q : cs.aq) ev(PolyRef{R_POLY, (uint32_t)q.first}, q.second);
  for (auto& q : cs.fq) ev(PolyRef{R_SHPOLY, (uint32_t)q.first}, q.second);
  ev(PolyRef{R_RANDPOLY, 0}, 0);
  for (uint32_t j = 0; j < pk.M; ++j) ev(PolyRef{R_SHPOLY, cs.F + j}, 0);
  for (uint32_t s = 0; s < pk.nsets; ++s) {
    ev(PolyRef{R_POLY, pk.slot_pz(s)}, 0); ev(PolyRef{R_POLY, pk.slot_pz(s)}, 1);
    if (s + 1 != pk.nsets) ev(PolyRef{R_POLY, pk.slot_pz(s)}, last_rot);
  }
  for (uint32_t l = 0; l < pk.L; ++l) {
    ev(PolyRef{R_POLY, pk.slot_lk(l, 2)}, 0); ev(PolyRef{R_POLY, pk.slot_lk(l, 2)}, 1);
    ev(PolyRef{R_POLY, pk.slot_lk(l, 0)}, 0); ev(PolyRef{R_POLY, pk.slot_lk(l, 0)}, -1);
    ev(PolyRef{R_POLY, pk.slot_lk(l, 1)}, 0);
  }
  BZ_CHECK(pk.evals.size() == pk.nev, "internal: evaluation list mismatch");
  build_programs(pk);
}

}  // namespace bz

extern "C" {

static int pk_create_impl(bz_ctx* ctx, bz_params* params, const bz_circuit* cin, const void* fixed_values, const void* sigma_values,
                          const uint32_t* mapping, bz_pk** out) {
  PV_TRY(ctx, {
    BZ_CHECK(out && params && cin, "null argument");
    *out = nullptr;
    BZ_CHECK(params->p.curve == 0, "prover: only the Vesta commitment curve (circuits over pallas::Base) is wired up");
    BZ_CHECK(cin->k == params->p.k, "circuit k != params k");
    std::unique_ptr<bz_pk> h(new bz_pk());
    PkImpl& pk = h->p;
    pk.params = &params->p;
    const bzh::Field& F = C->fp;
    pk_host_setup(C->fp, pk, cin);
    const CircuitCopy& cs = pk.cs;
    const uint32_t n = pk.n, en = pk.ext_n;
    cudaStream_t st = C->stream;
    // ---- Lagrange images, polys, cosets
    const uint32_t FM = cs.F + pk.M;
    pk.lval.alloc((size_t)std::max(1u, FM) * n * 32);
    if (cs.F) BZ_CUDA(cudaMemcpyAsync(pk.lval.p, fixed_values, (size_t)cs.F * n * 32, cudaMemcpyHostToDevice, st));
    pk.omega_pows.alloc((size_t)n * 32);
    geometric_kernel<FpP><<<(n + 127) / 128, 128, 0, st>>>((DFe*)pk.omega_pows.p, dfe(F.one()), dfe(pk.omega), n);
    C->kernel_launches++;
    if (pk.M && sigma_values) BZ_CUDA(cudaMemcpyAsync((char*)pk.lval.p + (size_t)cs.F * n * 32, sigma_values, (size_t)pk.M * n * 32, cudaMemcpyHostToDevice, st));
    else if (pk.M) {
      BZ_CHECK(mapping, "neither sigma values nor a permutation mapping given");
      const uint64_t total = (uint64_t)pk.M * n;
      for (uint64_t i = 0; i < total; ++i) BZ_CHECK(mapping[2 * i] < pk.M && mapping[2 * i + 1] < n, "permutation mapping out of range");
      DevBuf d_map, d_delta;
      d_map.alloc(total * 8); d_delta.alloc((size_t)pk.M * 32);
      BZ_CUDA(cudaMemcpyAsync(d_map.p, mapping, total * 8, cudaMemcpyHostToDevice, st));
      geometric_kernel<FpP><<<(pk.M + 127) / 128, 128, 0, st>>>((DFe*)d_delta.p, dfe(F.one()), dfe(F.delta()), pk.M);
      sigma_from_mapping_kernel<FpP><<<(unsigned)((total + 127) / 128), 128, 0, st>>>((const uint32_t*)d_map.p, (const DFe*)pk.omega_pows.p, (const DFe*)d_delta.p,
                                                                                    (DFe*)pk.lval.p + (size_t)cs.F * n, total);
      C->kernel_launches += 2;
      BZ_CUDA(cudaStreamSynchronize(st));
    }
    const uint32_t ND = (uint32_t)pk.derived.size();
    pk.shpoly.alloc((size_t)std::max(1u, FM) * n * 32);
    pk.shcoset.alloc((size_t)(FM + 5 + ND) * en * 32);
    NttFusion inv; inv.post_mode = 1;
    NttFusion ext; ext.n_in = pk.ext_k > cs.k ? n : 0; ext.pre_zeta = true;
    if (FM) {
      ntt_run(C, 0, pk.lval.p, pk.shpoly.p, cs.k, true, FM, inv);
      ntt_run(C, 0, pk.shpoly.p, pk.shcoset.p, pk.ext_k, false, FM, ext);
    }
    {  // l0, l_blind, l_last, active
      std::vector<HFe> tmp((size_t)4 * n, F.zero());
      tmp[0] = F.one();
      for (uint32_t i = n - cs.bf; i < n; ++i) tmp[(size_t)n + i] = F.one();
      tmp[(size_t)2 * n + (n - cs.bf - 1)] = F.one();
      for (uint32_t i = 0; i < n - cs.bf - 1; ++i) tmp[(size_t)3 * n + i] = F.one();
      DevBuf d_l, d_p;
      d_l.alloc((size_t)4 * n * 32); d_p.alloc((size_t)4 * n * 32);
      BZ_CUDA(cudaMemcpyAsync(d_l.p, tmp.data(), (size_t)4 * n * 32, cudaMemcpyHostToDevice, st));
      ntt_run(C, 0, d_l.p, d_p.p, cs.k, true, 4, inv);
      ntt_run(C, 0, d_p.p, (char*)pk.shcoset.p + (size_t)FM * en * 32, pk.ext_k, false, 4, ext);
      BZ_CUDA(cudaStreamSynchronize(st));
    }
    geometric_kernel<FpP><<<(en + 127) / 128, 128, 0, st>>>((DFe*)pk.shcoset.p + (size_t)(FM + 4) * en, dfe(F.zeta()), dfe(pk.ext_omega), en);
    C->kernel_launches += 1;
    if (ND) {  // derived shared columns: the fixed-only sub-expressions of the gates on the extended coset, once per key
      ProgBuilder pb; pb.scale = 1 << (pk.ext_k - cs.k);
      for (uint32_t j = 0; j < ND; ++j) { emit_tokens(pb, cs, pk.derived[j].tokens, 0, (uint32_t)pk.derived[j].tokens.size()); pb.store(j); }
      BZ_CHECK(pb.max_depth <= EVAL_STACK, "fixed sub-expression too deep for the evaluator stack");
      BZ_CHECK(pb.code.size() * 4 <= 96 * 1024, "fixed sub-expression program too large for shared memory");
      DevBuf d_code, d_rot, d_consts;
      d_code.alloc(pb.code.size() * 4); d_rot.alloc(std::max<size_t>(1, pb.rot_table.size()) * 4); d_consts.alloc(std::max<size_t>(1, cs.consts.size()) * 32);
      BZ_CUDA(cudaMemcpyAsync(d_code.p, pb.code.data(), pb.code.size() * 4, cudaMemcpyHostToDevice, st));
      if (!pb.rot_table.empty()) BZ_CUDA(cudaMemcpyAsync(d_rot.p, pb.rot_table.data(), pb.rot_table.size() * 4, cudaMemcpyHostToDevice, st));
      if (!cs.consts.empty()) BZ_CUDA(cudaMemcpyAsync(d_consts.p, cs.consts.data(), cs.consts.size() * 32, cudaMemcpyHostToDevice, st));
      EvalArgs<FpP> a{};
      a.code = (const uint32_t*)d_code.p; a.n_instr = (uint32_t)pb.code.size(); a.logN = pk.ext_k; a.rot = (const int32_t*)d_rot.p;
      a.pbase = nullptr; a.pstride = 0; a.sbase = (const DFe*)pk.shcoset.p; a.consts = (const DFe*)d_consts.p; a.cstride = 0;
      a.out = (DFe*)pk.shcoset.p + (size_t)(FM + 5) * en; a.ostride = 0; a.tev = nullptr; a.tn = 1;
      static PerDeviceOnce once;
      once.run(C->device, [] { cudaFuncSetAttribute(eval_program_kernel<FpP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024); });
      eval_program_kernel<FpP><<<dim3((en + 127) / 128, 1), 128, pb.code.size() * 4, st>>>(a);
      C->kernel_launches++;
      BZ_CUDA(cudaGetLastError());
      BZ_CUDA(cudaStreamSynchronize(st));
    }
    {  // t_evaluations
      uint32_t tn = 1u << (pk.ext_k - cs.k);
      HFe orig = F.pow_u64(F.zeta(), n), step = F.pow_u64(pk.ext_omega, n), cur = orig;
      std::vector<HFe> t;
      for (uint32_t i = 0; i < tn; ++i) { t.push_back(F.inv(F.sub(cur, F.one()))); cur = F.mul(cur, step); }
      pk.tev.alloc((size_t)tn * 32);
      BZ_CUDA(cudaMemcpyAsync(pk.tev.p, t.data(), (size_t)tn * 32, cudaMemcpyHostToDevice, st));
      BZ_CUDA(cudaStreamSynchronize(st));
    }
    pk.d_evals.alloc(pk.evals.size() * sizeof(EvalQuery));
    BZ_CUDA(cudaMemcpy(pk.d_evals.p, pk.evals.data(), pk.evals.size() * sizeof(EvalQuery), cudaMemcpyHostToDevice));
    upload_programs(pk);
    BZ_CUDA(cudaStreamSynchronize(st));
    *out = h.release();
  });
}

API int bz_pk_create(bz_ctx* ctx, bz_params* params, const bz_circuit* cin, const void* fixed_values, const void* sigma_values, bz_pk** out) {
  if (!ctx) return BZ_ERR_INVALID;
  if (cin && cin->n_perm_columns && !sigma_values) { ctx->c.last_error = "null sigma_values"; return BZ_ERR_INVALID; }
  return pk_create_impl(ctx, params, cin, fixed_values, sigma_values, nullptr, out);
}
API int bz_pk_create_from_assembly(bz_ctx* ctx, bz_params* params, const bz_circuit* cin, const void* fixed_values, const uint32_t* mapping, bz_pk** out) {
  if (!ctx) return BZ_ERR_INVALID;
  return pk_create_impl(ctx, params, cin, fixed_values, nullptr, mapping, out);
}

// keygen_vk's commitments: commit_lagrange(column, Blind::default() = 1) for every fixed and every sigma column
API int bz_pk_vk_commitments(bz_ctx* ctx, bz_pk* pkh, void* fixed_commitments, void* perm_commitments) {
  PV_TRY(ctx, {
    BZ_CHECK(pkh, "null argument");
    PkImpl& pk = pkh->p;
    const uint32_t FM = pk.cs.F + pk.M, n = pk.n;
    if (FM && pk.vk_fixed_comm.size() + pk.vk_perm_comm.size() != (size_t)FM * 8) {
      cudaStream_t st = C->stream;
      std::vector<void*> mainp(FM), extrap(FM);
      DevBuf &d_out = C->stage[1], &d_extra = C->stage[3], &d_ptrs = C->stage[4];
      d_extra.ensure((size_t)FM * 64); d_out.ensure((size_t)FM * 64);
      std::vector<HFe> ex((size_t)FM * 2, C->fp.zero());
      for (uint32_t j = 0; j < FM; ++j) { mainp[j] = (DFe*)pk.lval.p + (size_t)j * n; extrap[j] = (DFe*)d_extra.p + (size_t)j * 2; ex[2 * j] = C->fp.one(); }
      BZ_CUDA(cudaMemcpyAsync(d_extra.p, ex.data(), ex.size() * 32, cudaMemcpyHostToDevice, st));
      const void* const* d = upload_msm_ptrs(C, d_ptrs, mainp, extrap);
      params_commit_run(C, *pk.params, true, d, d + FM, FM, d_out.p);
      std::vector<uint64_t> all((size_t)FM * 8);
      BZ_CUDA(cudaMemcpyAsync(all.data(), d_out.p, all.size() * 8, cudaMemcpyDeviceToHost, st));
      BZ_CUDA(cudaStreamSynchronize(st));
      pk.vk_fixed_comm.assign(all.begin(), all.begin() + (size_t)pk.cs.F * 8);
      pk.vk_perm_comm.assign(all.begin() + (size_t)pk.cs.F * 8, all.end());
    }
    if (fixed_commitments && pk.cs.F) memcpy(fixed_commitments, pk.vk_fixed_comm.data(), pk.vk_fixed_comm.size() * 8);
    if (perm_commitments && pk.M) memcpy(perm_commitments, pk.vk_perm_comm.data(), pk.vk_perm_comm.size() * 8);
  });
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------------
namespace bz {

struct Prover {
  Ctx* C; PkImpl& pk; uint32_t B;
  const bzh::Field& F; const bzh::Field& Fq;
  cudaStream_t st;
  PkImpl::Work& w;
  Regions reg;
  std::vector<ProofState> ps;
  uint32_t n, en, k;
  size_t desc_off = 0;

  Prover(Ctx* c, PkImpl& p, uint32_t b) : C(c), pk(p), B(b), F(c->fp), Fq(c->fq), st(c->stream), w(p.work), ps(b) {
    n = pk.n; en = pk.ext_n; k = pk.cs.k;
    memset(&reg, 0, sizeof(reg));
    reg.base[R_VAL] = w.val.p; reg.stride[R_VAL] = (uint64_t)pk.NS * n;
    reg.base[R_POLY] = w.poly.p; reg.stride[R_POLY] = (uint64_t)pk.NS * n;
    reg.base[R_MISC] = w.misc.p; reg.stride[R_MISC] = (uint64_t)pk.NM * n;
    reg.base[R_RANDPOLY] = (DFe*)w.rnd.p + pk.r_randpoly; reg.stride[R_RANDPOLY] = pk.R;
    reg.base[R_SPOLY] = (DFe*)w.rnd.p + pk.r_spoly; reg.stride[R_SPOLY] = pk.R;
    reg.base[R_SHPOLY] = pk.shpoly.p; reg.stride[R_SHPOLY] = 0;
    reg.base[R_SHVAL] = pk.lval.p; reg.stride[R_SHVAL] = 0;
    reg.base[R_HCOEF] = w.hcoef.p; reg.stride[R_HCOEF] = en;
  }

  DFe* val(uint32_t b, uint32_t slot) { return (DFe*)w.val.p + ((uint64_t)b * pk.NS + slot) * n; }
  DFe* polyp(uint32_t b, uint32_t slot) { return (DFe*)w.poly.p + ((uint64_t)b * pk.NS + slot) * n; }
  DFe* misc(uint32_t b, uint32_t slot) { return (DFe*)w.misc.p + ((uint64_t)b * pk.NM + slot) * n; }
  DFe* rnd(uint32_t b, uint32_t idx) { return (DFe*)w.rnd.p + (uint64_t)b * pk.R + idx; }

  // small descriptor arena in device memory (reset per phase)
  template <class T> T* upload_desc(const std::vector<T>& v) {
    size_t bytes = v.size() * sizeof(T);
    desc_off = (desc_off + 15) & ~size_t(15);
    BZ_CHECK(desc_off + bytes <= w.descs.bytes, "descriptor arena overflow");
    T* d = (T*)((char*)w.descs.p + desc_off);
    BZ_CUDA(cudaMemcpyAsync(d, v.data(), bytes, cudaMemcpyHostToDevice, st));
    desc_off += bytes;
    return d;
  }

  void upload_consts() {
    std::vector<HFe> all((size_t)B * pk.cstride);
    for (uint32_t b = 0; b < B; ++b) memcpy(&all[(size_t)b * pk.cstride], ps[b].consts.data(), (size_t)pk.cstride * 32);
    BZ_CUDA(cudaMemcpyAsync(w.consts.p, all.data(), all.size() * 32, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaStreamSynchronize(st));       // `all` goes out of scope
  }

  // ---- batched NTT helpers over slot ranges ----
  void to_coeff(uint32_t slot0, uint32_t count) {
    NttFusion fu; fu.post_mode = 1;
    ntt_run(C, 0, val(0, slot0), polyp(0, slot0), k, true, count, fu, B, (uint64_t)pk.NS * n, (uint64_t)pk.NS * n);
  }
  void to_coset(uint32_t slot0, uint32_t count) {
    NttFusion fu; fu.n_in = pk.ext_k > k ? n : 0; fu.pre_zeta = true;
    ntt_run(C, 0, polyp(0, slot0), (DFe*)w.coset.p + (uint64_t)slot0 * en, pk.ext_k, false, count, fu, B, (uint64_t)pk.NS * n, (uint64_t)pk.NS * en);
  }

  // ---- commitments: a list of (main poly device ptr fn, blind) per proof; results host-side ----
  struct CommitReq { PolyRef poly; bool lagrange; };
  // commits reqs (same list for every proof); blinds[b][i] host scalars for point w.  Output points[b][i].
  void commit(const std::vector<CommitReq>& reqs, const std::vector<std::vector<HFe>>& blinds, std::vector<std::vector<HostPoint>>& pts,
              const std::vector<std::array<HFe, 2>>* extras_full = nullptr) {
    const uint32_t nr = (uint32_t)reqs.size();
    pts.assign(B, std::vector<HostPoint>(nr));
    // all requests of one call share the basis
    bool lag = reqs[0].lagrange;
    std::vector<void*> mainp((size_t)B * nr), extrap((size_t)B * nr);
    std::vector<HFe> ex((size_t)B * nr * 2, F.zero());
    BZ_CHECK((size_t)B * nr * 2 * 32 <= w.extras.bytes && (size_t)B * nr * 2 * sizeof(void*) <= w.ptrs.bytes && (size_t)B * nr * 128 <= w.commits.bytes,
             "commit batch too large for the workspace");
    for (uint32_t b = 0; b < B; ++b)
      for (uint32_t i = 0; i < nr; ++i) {
        BZ_CHECK(reqs[i].lagrange == lag, "mixed bases in one commit batch");
        size_t j = (size_t)b * nr + i;
        uint64_t len = n;
        mainp[j] = (DFe*)reg.base[reqs[i].poly.kind] + (uint64_t)b * reg.stride[reqs[i].poly.kind] + (uint64_t)reqs[i].poly.slot * len;
        extrap[j] = (DFe*)w.extras.p + j * 2;
        if (extras_full) { ex[j * 2] = (*extras_full)[j][0]; ex[j * 2 + 1] = (*extras_full)[j][1]; }
        else ex[j * 2] = blinds[b][i];
      }
    BZ_CUDA(cudaMemcpyAsync(w.extras.p, ex.data(), ex.size() * 32, cudaMemcpyHostToDevice, st));
    uint32_t n_msm = B * nr;
    run_msms(lag, mainp, extrap, n_msm);
    read_points(n_msm, nr, pts);
  }
  // one batch of commitments into w.commits: the table MSM's XYZZ sums, or affine points from the bucket MSM (read_points)
  void run_msms(bool lagrange, const std::vector<void*>& mainp, const std::vector<void*>& extrap, uint32_t n_msm) {
    const ParamsImpl& pr = *pk.params;
    const uint32_t world = C->shard_world, rank = C->shard_rank;
    const void* const* dm = upload_msm_ptrs(C, w.ptrs, mainp, extrap);
    const void* const* de = dm + n_msm;
    if (world > 1 && pr.use_tables && n_msm >= world) {
      // one large proof across GPUs, table path: rank r sums the contiguous MSMs [r * per, (r + 1) * per) and the 128-byte
      // XYZZ results are all-gathered (every rank holds the same tables); fewer MSMs than ranks are computed redundantly
      const uint32_t per = (n_msm + world - 1) / world, lo = std::min(n_msm, rank * per), hi = std::min(n_msm, lo + per);
      BZ_CHECK((size_t)per * 128 <= C->shard_cap, "sharding exchange buffer too small");
      BZ_CUDA(cudaMemsetAsync(C->shard_send, 0, (size_t)per * 128, st));
      if (hi > lo) params_commit_run(C, pr, lagrange, dm + lo, de + lo, hi - lo, C->shard_send, true);
      if (C->shard_exchange(C->shard_user, (size_t)per * 128) != 0) throw Error(BZ_ERR_CUDA, "sharding: all-gather callback failed");
      BZ_CUDA(cudaMemcpyAsync(w.commits.p, C->shard_recv, (size_t)n_msm * 128, cudaMemcpyDeviceToDevice, st));
      return;
    }
    if (world > 1 && !pr.use_tables) {
      const uint32_t npts = (lagrange ? pr.fb_gl : pr.fb_g).npts;
      const void* bases = lagrange ? pr.gl_w.p : pr.g_w_u.p;
      if (n_msm >= world) {
        // column deal: rank r owns the contiguous MSMs [r * per, (r + 1) * per); one all-gather of per x 96 B per rank
        const uint32_t per = (n_msm + world - 1) / world, lo = std::min(n_msm, rank * per), hi = std::min(n_msm, lo + per);
        BZ_CHECK((size_t)per * 96 <= C->shard_cap, "sharding exchange buffer too small");
        BZ_CUDA(cudaMemsetAsync(C->shard_send, 0, (size_t)per * 96, st));
        msm_run_batch(C, pr.curve, dm + lo, de + lo, n, 0, npts, bases, hi - lo, C->shard_send);
        if (C->shard_exchange(C->shard_user, (size_t)per * 96) != 0) throw Error(BZ_ERR_CUDA, "sharding: all-gather callback failed");
        jac_to_affine_run(C, pr.curve, C->shard_recv, w.commits.p, n_msm);          // rank-major = MSM order
        return;
      }
      // fewer MSMs than ranks (random polynomial, q', S, the two IPA terms): every MSM split by point range, the partials summed
      BZ_CHECK((size_t)n_msm * 96 <= C->shard_cap, "sharding exchange buffer too small");
      const uint32_t base = npts / world, rem = npts % world, plo = rank * base + std::min(rank, rem), cnt = base + (rank < rem ? 1u : 0u);
      msm_run_batch(C, pr.curve, dm, de, n, plo, cnt, (const char*)bases + (size_t)plo * 64, n_msm, C->shard_send);
      if (C->shard_exchange(C->shard_user, (size_t)n_msm * 96) != 0) throw Error(BZ_ERR_CUDA, "sharding: all-gather callback failed");
      w.msm_jac.ensure((size_t)n_msm * world * 96);
      for (uint32_t j = 0; j < n_msm; ++j) {
        // partials of MSM j sit at recv[r][j]: gather them contiguously, then one kernel adds them and normalises
        BZ_CUDA(cudaMemcpy2DAsync((char*)w.msm_jac.p + (size_t)j * world * 96, 96, (const char*)C->shard_recv + (size_t)j * 96, (size_t)n_msm * 96, 96, world, cudaMemcpyDeviceToDevice, st));
        jac_sum_run(C, pr.curve, (const char*)w.msm_jac.p + (size_t)j * world * 96, world, (char*)w.commits.p + (size_t)j * 64);
      }
      return;
    }
    params_commit_run(C, pr, lagrange, dm, de, n_msm, w.commits.p, pr.use_tables);
  }
  // Commitments come back unnormalised from the table MSM (XYZZ, 128 B): one batched inversion on the host for the
  // whole call (Montgomery's trick, ~9 host multiplications per point) instead of a single-thread Fermat chain per
  // commitment on the device (~0.1 ms of latency per launch).  The bucket-MSM path (large k) returns affine points.
  void read_points(uint32_t n_msm, uint32_t nr, std::vector<std::vector<HostPoint>>& pts, bool force_affine = false) {
    const bool xyzz = pk.params->use_tables && !force_affine;
    BZ_CUDA(cudaMemcpyAsync(w.h_pinned, w.commits.p, (size_t)n_msm * (xyzz ? 128 : 64), cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
    const uint64_t* h = (const uint64_t*)w.h_pinned;
    if (!xyzz) {
      for (uint32_t b = 0; b < B; ++b)
        for (uint32_t i = 0; i < nr; ++i) affine_to_host(Fq, h + ((size_t)b * nr + i) * 8, pts[b][i]);
      return;
    }
    std::vector<HFe> zi3(n_msm);                       // zzz, then 1 / zzz (0 for the identity)
    for (uint32_t j = 0; j < n_msm; ++j) memcpy(zi3[j].l, h + (size_t)j * 16 + 12, 32);
    host_batch_invert(Fq, zi3);
    for (uint32_t j = 0; j < n_msm; ++j) {
      HFe x, y, zz;
      memcpy(x.l, h + (size_t)j * 16, 32); memcpy(y.l, h + (size_t)j * 16 + 4, 32); memcpy(zz.l, h + (size_t)j * 16 + 8, 32);
      HostPoint& p = pts[j / nr][j % nr];
      if (zi3[j].is_zero()) { p.identity = true; memset(p.x, 0, 32); memset(p.y, 0, 32); continue; }
      const HFe t = Fq.mul(zz, zi3[j]), zi2 = Fq.sqr(t);  // (zz / zzz)^2 = 1 / zz
      p.identity = false;
      Fq.to_repr(Fq.mul(x, zi2), p.x); Fq.to_repr(Fq.mul(y, zi3[j]), p.y);
    }
  }

  void launch_copy(const std::vector<CopyDesc>& d, uint64_t len) {
    if (d.empty()) return;
    CopyDesc* dd = upload_desc(d);
    copy_rows_kernel<FpP><<<dim3((unsigned)d.size(), B), 64, 0, st>>>(reg, len, dd, (const DFe*)w.rnd.p, pk.R);
    C->kernel_launches++;
  }

  void grand_product(PolyRef zref, bool has_z0, PolyRef z0ref, uint32_t z0_index) {
    DFe* num = (DFe*)w.nd.p; DFe* den = num + (uint64_t)B * n; DFe* pnum = den + (uint64_t)B * n; DFe* sden = pnum + (uint64_t)B * n;
    ProfScope prof(C, PROF_SCAN);
    const uint32_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (ntiles <= 8) {          // Shot / Board: one CTA per proof walks the 1-2 tiles
      product_scan_kernel<FpP><<<dim3(1, B), SCAN_THREADS, 0, st>>>(num, pnum, n, n, 0);
      product_scan_kernel<FpP><<<dim3(1, B), SCAN_THREADS, 0, st>>>(den, sden, n, n, 1);
    } else {                    // large domains: tile products, scan of the tile products, rescan with carry-in
      BZ_CHECK(ntiles <= (uint32_t)SCAN_TILE, "grand product: domain too large for the two-level scan");
      w.scan_tmp.ensure((size_t)4 * B * ntiles * 32);
      DFe* tot_n = (DFe*)w.scan_tmp.p; DFe* car_n = tot_n + (size_t)B * ntiles; DFe* tot_d = car_n + (size_t)B * ntiles; DFe* car_d = tot_d + (size_t)B * ntiles;
      product_scan_kernel<FpP><<<dim3(ntiles, B), SCAN_THREADS, 0, st>>>(num, pnum, n, n, 0, 1u, nullptr, tot_n);
      product_scan_kernel<FpP><<<dim3(ntiles, B), SCAN_THREADS, 0, st>>>(den, sden, n, n, 1, 1u, nullptr, tot_d);
      product_scan_kernel<FpP><<<dim3(1, B), SCAN_THREADS, 0, st>>>(tot_n, car_n, ntiles, ntiles, 0);
      product_scan_kernel<FpP><<<dim3(1, B), SCAN_THREADS, 0, st>>>(tot_d, car_d, ntiles, ntiles, 0);
      product_scan_kernel<FpP><<<dim3(ntiles, B), SCAN_THREADS, 0, st>>>(num, pnum, n, n, 0, 1u, car_n, nullptr);
      product_scan_kernel<FpP><<<dim3(ntiles, B), SCAN_THREADS, 0, st>>>(den, sden, n, n, 1, 1u, car_d, nullptr);
      C->kernel_launches += 4;
    }
    grand_product_finish_kernel<FpP><<<dim3((n + 127) / 128, B), 128, 0, st>>>(pnum, sden, n, reg, zref, n, z0ref, z0_index, has_z0 ? 1 : 0);
    C->kernel_launches += 3;
  }

  // Horner evaluation of nq polynomials per proof into w.evalout[b * nq + q]
  void eval_launch(const EvalQuery* d_queries, uint32_t nq) {
    const uint32_t splits = std::max(1u, n / 16384u);        // large domains: several CTAs per (query, proof)
    if (splits == 1) eval_queries_kernel<FpP><<<dim3(nq, B), EVALQ_THREADS, 0, st>>>(reg, n, d_queries, (const DFe*)w.consts.p, pk.cstride, (DFe*)w.evalout.p, nq);
    else {
      w.eval_tmp.ensure((size_t)B * nq * splits * 32);
      eval_queries_kernel<FpP><<<dim3(nq, B, splits), EVALQ_THREADS, 0, st>>>(reg, n, d_queries, (const DFe*)w.consts.p, pk.cstride, (DFe*)w.eval_tmp.p, nq);
      eval_reduce_kernel<FpP><<<(B * nq + 127) / 128, 128, 0, st>>>((const DFe*)w.eval_tmp.p, splits, (DFe*)w.evalout.p, B * nq);
      C->kernel_launches++;
    }
    C->kernel_launches++;
  }
  void evaluate(const EvalQuery* d_queries, uint32_t nq, std::vector<std::vector<HFe>>& out) {
    {
      ProfScope prof(C, PROF_EVAL);
      eval_launch(d_queries, nq);
    }
    BZ_CUDA(cudaMemcpyAsync(w.h_pinned, w.evalout.p, (size_t)B * nq * 32, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
    out.assign(B, std::vector<HFe>(nq));
    for (uint32_t b = 0; b < B; ++b) memcpy(out[b].data(), (char*)w.h_pinned + (size_t)b * nq * 32, (size_t)nq * 32);
  }

  void lincomb(const std::vector<LinCombDesc>& descs, const std::vector<PolyRef>& refs) {
    LinCombDesc* dd = upload_desc(descs);
    PolyRef* dr = upload_desc(refs);
    ProfScope prof(C, PROF_POLY);
    lincomb_kernel<FpP><<<dim3((n + 127) / 128, B, (unsigned)descs.size()), 128, 0, st>>>(reg, n, dd, dr, (const DFe*)w.consts.p, pk.cstride);
    C->kernel_launches++;
  }

  void compute_h();
  void run(const void* instances, const uint32_t* instance_lens, uint32_t instance_stride, const void* advice, const void* rand_wide, uint8_t* proofs);
};

// steps 11-12 up to the coefficients of h(X): w.coset (all slots) + the per-proof constants -> w.hcoef[b][0 .. ext_n)
// (the quotient program, the fused division by t(X), the inverse NTTs of the three degree tiers)
void Prover::compute_h() {
    EvalArgs<FpP> a{};
    a.code = (const uint32_t*)pk.q_code[0].p; a.n_instr = pk.q_ninstr[0]; a.logN = pk.ext_k; a.rot = (const int32_t*)pk.q_rot[0].p;
    a.pbase = (const DFe*)w.coset.p; a.pstride = (uint64_t)pk.NS * en; a.sbase = (const DFe*)pk.shcoset.p;
    a.consts = (const DFe*)w.consts.p; a.cstride = pk.cstride;
    a.out = (DFe*)w.hext.p; a.ostride = en; a.tev = (const DFe*)pk.tev.p; a.tn = 1u << (pk.ext_k - k);
    static PerDeviceOnce once;
    once.run(C->device, [] { cudaFuncSetAttribute(eval_program_kernel<FpP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024); });
    // One large proof across GPUs: every rank evaluates a contiguous range of the extended-coset points of each tier and the
    // ranges are exchanged with one all-gather (32 B per point) -- h(X) is point-wise, so the evaluation shards perfectly.
    // Only for a batch of one (the slices of a batch would be strided) and when the exchange buffers were sized for it.
    const uint32_t world = C->shard_world, rank = C->shard_rank;
    uint64_t slice_bytes = 0;
    for (uint32_t t = 0; t < PkImpl::Q_TIERS; ++t) if (t == 0 || pk.q_ninstr[t]) slice_bytes += (uint64_t)(en >> t) / std::max(1u, world) * 32;
    const bool split = world > 1 && B == 1 && (en >> (PkImpl::Q_TIERS - 1)) >= 128u * world && (en >> (PkImpl::Q_TIERS - 1)) % world == 0 && slice_bytes <= C->shard_cap;
    {
      ProfScope prof(C, PROF_QUOTIENT);
      auto launch = [&](uint32_t t, EvalArgs<FpP> args, uint32_t points) {
        if (split) { points /= world; args.first = rank * points; }
        const dim3 grid((points + 127) / 128, B);
        if (pk.q_gen[t]) pk.q_gen[t](args, grid, st);                   // circuit-specialised straight-line code (gen_quotient.cu)
        else eval_program_kernel<FpP><<<grid, 128, pk.q_ninstr[t] * 4, st>>>(args);
        C->kernel_launches++;
      };
      launch(0, a, en);
      DFe* low_out = (DFe*)w.hext_low.p;
      for (uint32_t t = 1; t < PkImpl::Q_TIERS; ++t) {      // lower-degree terms: every 2^t-th extended point
        if (!pk.q_ninstr[t]) continue;
        EvalArgs<FpP> al = a;
        al.code = (const uint32_t*)pk.q_code[t].p; al.n_instr = pk.q_ninstr[t]; al.rot = (const int32_t*)pk.q_rot[t].p;
        al.stride_log = t; al.out = low_out; al.ostride = en >> t;
        launch(t, al, en >> t);
        low_out += (size_t)B * (en >> t);
      }
    }
    if (split) {
      // send = [tier 0 slice | tier 1 slice | ...] of this rank; recv = the same layout of every rank, rank-major
      DFe* tier_out[PkImpl::Q_TIERS];
      uint32_t tier_pts[PkImpl::Q_TIERS];
      DFe* lo_ptr = (DFe*)w.hext_low.p;
      for (uint32_t t = 0; t < PkImpl::Q_TIERS; ++t) {
        tier_pts[t] = (t == 0 || pk.q_ninstr[t]) ? (en >> t) / world : 0;
        tier_out[t] = t == 0 ? (DFe*)w.hext.p : lo_ptr;
        if (t > 0 && pk.q_ninstr[t]) lo_ptr += (size_t)(en >> t);
      }
      size_t off = 0;
      for (uint32_t t = 0; t < PkImpl::Q_TIERS; ++t) {
        if (!tier_pts[t]) continue;
        BZ_CUDA(cudaMemcpyAsync((char*)C->shard_send + off, tier_out[t] + (size_t)rank * tier_pts[t], (size_t)tier_pts[t] * 32, cudaMemcpyDeviceToDevice, st));
        off += (size_t)tier_pts[t] * 32;
      }
      if (C->shard_exchange(C->shard_user, slice_bytes) != 0) throw Error(BZ_ERR_CUDA, "sharding: all-gather callback failed");
      for (uint32_t r = 0; r < world; ++r) {
        if (r == rank) continue;
        size_t o = (size_t)r * slice_bytes;
        for (uint32_t t = 0; t < PkImpl::Q_TIERS; ++t) {
          if (!tier_pts[t]) continue;
          BZ_CUDA(cudaMemcpyAsync(tier_out[t] + (size_t)r * tier_pts[t], (const char*)C->shard_recv + o, (size_t)tier_pts[t] * 32, cudaMemcpyDeviceToDevice, st));
          o += (size_t)tier_pts[t] * 32;
        }
      }
    }
    NttFusion fu; fu.post_mode = 3;
    ntt_run(C, 0, w.hext.p, w.hcoef.p, pk.ext_k, true, B, fu);
    {
      const DFe* low_in = (const DFe*)w.hext_low.p;
      for (uint32_t t = 1; t < PkImpl::Q_TIERS; ++t) {
        if (!pk.q_ninstr[t]) continue;
        ntt_run(C, 0, low_in, w.hcoef_low.p, pk.ext_k - t, true, B, fu);
        ProfScope prof(C, PROF_POLY);
        add_low_kernel<FpP><<<dim3(((en >> t) + 127) / 128, B), 128, 0, st>>>((DFe*)w.hcoef.p, en, (const DFe*)w.hcoef_low.p, en >> t);
        C->kernel_launches++;
        low_in += (size_t)B * (en >> t);
      }
    }
}

void Prover::run(const void* instances, const uint32_t* instance_lens, uint32_t instance_stride, const void* advice, const void* rand_wide, uint8_t* proofs) {
  const CircuitCopy& cs = pk.cs;
  const uint32_t G = cs.G, I = cs.I, L = pk.L, bf = cs.bf, usable = pk.usable;
  for (uint32_t i = 0; i < I; ++i) {
    if (instance_lens[i] > usable) throw Error(BZ_ERR_INVALID, "Error::InstanceTooLarge");
    BZ_CHECK(instance_lens[i] <= instance_stride, "instance_lens[i] exceeds instance_stride");
  }
  // ---- per-proof host state
  for (uint32_t b = 0; b < B; ++b) {
    ps[b].out = proofs + (size_t)b * pk.proof_size;
    memset(ps[b].out, 0, pk.proof_size);
    ps[b].wide = (const uint8_t*)rand_wide + (size_t)b * pk.R * 64;
    ps[b].blinds.assign(pk.nblinds, F.zero());
    ps[b].consts.assign(pk.cstride, F.zero());
    for (uint32_t i = 0; i < pk.NC; ++i) ps[b].consts[i] = cs.consts[i];
    ps[b].consts[pk.C_ONE] = F.one();
    t_common_scalar(ps[b], F, cs.vk_repr);                                     // step 0
  }
  // ---- upload: randomness (reduced on device), advice, instances.  Inputs may live in host or device memory
  // (cudaMemcpyDefault); blinds are re-derived on the host from the same RNG words, so a device-resident stream
  // is mirrored to the host once.
  // The host reads a few dozen words (blinds); the two n-word slices (random polynomial, the IPA's S polynomial) are only ever
  // used on the device, so only the three short ranges around them are mirrored (at k = 20 the whole stream is 134 MB and a
  // pageable copy of it cost 40 ms per proof).  The mirror keeps the stream's indexing; untouched pages are never committed.
  std::unique_ptr<uint8_t[]> wide_host;
  {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, rand_wide) == cudaSuccess && at.type == cudaMemoryTypeDevice) {
      wide_host.reset(new uint8_t[(size_t)B * pk.R * 64]);
      const uint32_t ranges[3][2] = {{0, pk.r_randpoly}, {pk.r_randpoly + n, pk.r_spoly}, {pk.r_spoly + n, pk.R}};
      for (const auto& rg : ranges)          // one strided copy per range: row b = proof b
        if (rg[1] > rg[0])
          BZ_CUDA(cudaMemcpy2DAsync(wide_host.get() + (size_t)rg[0] * 64, (size_t)pk.R * 64, (const uint8_t*)rand_wide + (size_t)rg[0] * 64, (size_t)pk.R * 64,
                                    (size_t)(rg[1] - rg[0]) * 64, B, cudaMemcpyDeviceToHost, st));
      BZ_CUDA(cudaStreamSynchronize(st));
      for (uint32_t b = 0; b < B; ++b) ps[b].wide = wide_host.get() + (size_t)b * pk.R * 64;
    } else cudaGetLastError();
  }
  if (rand_wide != w.wide.p)        // bz_create_proofs_seeded expands the stream in place
    BZ_CUDA(cudaMemcpyAsync(w.wide.p, rand_wide, (size_t)B * pk.R * 64, cudaMemcpyDefault, st));
  {
    uint64_t tot = (uint64_t)B * pk.R;
    from_u512_kernel<FpP><<<(unsigned)((tot + 127) / 128), 128, 0, st>>>((const uint32_t*)w.wide.p, (DFe*)w.rnd.p, tot);
    C->kernel_launches++;
  }
  BZ_CUDA(cudaMemsetAsync(w.val.p, 0, (size_t)B * pk.NS * n * 32, st));
  for (uint32_t b = 0; b < B; ++b) {
    BZ_CUDA(cudaMemcpyAsync(val(b, 0), (const char*)advice + (size_t)b * G * n * 32, (size_t)G * n * 32, cudaMemcpyDefault, st));
    for (uint32_t i = 0; i < I; ++i)
      if (instance_lens[i])
        BZ_CUDA(cudaMemcpyAsync(val(b, pk.slot_inst(i)), (const char*)instances + ((size_t)b * I + i) * instance_stride * 32,
                                (size_t)instance_lens[i] * 32, cudaMemcpyDefault, st));
  }
  std::unique_ptr<NvtxRange> phase;
  desc_off = 0;
  // ---- step 1: instance commitments (blind 1), absorbed
  phase.reset(); phase.reset(new NvtxRange("step 1-2: instance + advice commitments, NTTs"));
  std::vector<std::vector<HostPoint>> pts;
  // ---- steps 1-2: instance commitments (blind 1; absorbed, not written) and advice commitments (blinding rows, then one blind
  // per column) in ONE commitment batch: both are commit_lagrange and no challenge separates them
  {
    std::vector<CopyDesc> cd;
    for (uint32_t g = 0; g < G; ++g) cd.push_back(CopyDesc{PolyRef{R_VAL, g}, usable, pk.r_adv_rows + g * (bf + 1), bf + 1});
    launch_copy(cd, n);
    std::vector<CommitReq> reqs;
    for (uint32_t i = 0; i < I; ++i) reqs.push_back({PolyRef{R_VAL, pk.slot_inst(i)}, true});
    for (uint32_t g = 0; g < G; ++g) reqs.push_back({PolyRef{R_VAL, g}, true});
    std::vector<std::vector<HFe>> bl(B, std::vector<HFe>(I + G, F.one()));
    for (uint32_t b = 0; b < B; ++b) for (uint32_t g = 0; g < G; ++g) { bl[b][I + g] = rnd_host(ps[b], F, pk.r_adv_blind + g); ps[b].blinds[g] = bl[b][I + g]; }
    commit(reqs, bl, pts);
    for (uint32_t b = 0; b < B; ++b) {
      for (uint32_t i = 0; i < I; ++i) t_common_point(ps[b], pts[b][i]);
      for (uint32_t g = 0; g < G; ++g) t_write_point(ps[b], pts[b][I + g]);
    }
    to_coeff(0, G + I);
    to_coset(0, G + I);
  }
  // ---- step 3
  for (uint32_t b = 0; b < B; ++b) ps[b].consts[pk.C_THETA] = t_squeeze(ps[b], F);
  upload_consts();
  // ---- steps 4-5: lookups
  phase.reset(); phase.reset(new NvtxRange("steps 4-5: lookup compression, permutation, commitments"));
  if (L) {
    {
      EvalArgs<FpP> a{};
      a.code = (const uint32_t*)pk.lk_code.p; a.n_instr = pk.lk_ninstr; a.logN = k; a.rot = (const int32_t*)pk.lk_rot.p;
      a.pbase = (const DFe*)w.val.p; a.pstride = (uint64_t)pk.NS * n; a.sbase = (const DFe*)pk.lval.p;
      a.consts = (const DFe*)w.consts.p; a.cstride = pk.cstride;
      a.out = misc(0, pk.m_cin0); a.ostride = (uint64_t)pk.NM * n; a.tev = nullptr; a.tn = 1;
      ProfScope prof(C, PROF_QUOTIENT);
      eval_program_kernel<FpP><<<dim3((n + 127) / 128, B), 128, pk.lk_ninstr * 4, st>>>(a);
      C->kernel_launches++;
    }
    if (n > LKP_MAX_N) {
      // large domains: device-wide radix sort / scans per (proof, lookup) (lookup.cu)
      BZ_CUDA(cudaMemsetAsync(w.lk_err.p, 0, (size_t)B * 4, st));
      ProfScope prof(C, PROF_SCAN);
      for (uint32_t b = 0; b < B; ++b)
        for (uint32_t l = 0; l < L; ++l)
          lookup_permute_large_run(C, misc(b, pk.m_cin0 + 2 * l), misc(b, pk.m_cin0 + 2 * l + 1), val(b, pk.slot_lk(l, 0)), val(b, pk.slot_lk(l, 1)), usable, (uint32_t*)w.lk_err.p + b);
      BZ_CUDA(cudaMemcpyAsync(w.h_err, w.lk_err.p, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    } else {
      // device: sort / permute (U: lookup/prover.rs::permute_expression_pair), one CTA per (lookup, proof)
      static PerDeviceOnce once;
      once.run(C->device, [] { cudaFuncSetAttribute(lookup_permute_kernel<FpP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lookup_permute_smem(LKP_MAX_N)); });
      std::vector<LookupPermDesc> pd;
      for (uint32_t l = 0; l < L; ++l)
        pd.push_back(LookupPermDesc{PolyRef{R_MISC, pk.m_cin0 + 2 * l}, PolyRef{R_MISC, pk.m_cin0 + 2 * l + 1}, PolyRef{R_VAL, pk.slot_lk(l, 0)}, PolyRef{R_VAL, pk.slot_lk(l, 1)}});
      LookupPermDesc* dpd = upload_desc(pd);
      BZ_CUDA(cudaMemsetAsync(w.lk_err.p, 0, (size_t)B * 4, st));
      {
        ProfScope prof(C, PROF_SCAN);
        lookup_permute_kernel<FpP><<<dim3(L, B), LKP_THREADS, lookup_permute_smem(n), st>>>(reg, n, usable, dpd, (DFe*)w.lk_sorted.p, (uint32_t*)w.lk_err.p);
        C->kernel_launches++;
      }
      BZ_CUDA(cudaMemcpyAsync(w.h_err, w.lk_err.p, (size_t)B * 4, cudaMemcpyDeviceToHost, st));     // read after the commitments' sync below
    }
    std::vector<CopyDesc> cd;
    std::vector<CommitReq> reqs;
    std::vector<std::vector<HFe>> bl(B, std::vector<HFe>(2 * L));
    for (uint32_t l = 0; l < L; ++l) {
      uint32_t r0 = pk.r_lk0 + l * (2 * (bf + 1) + 2);
      cd.push_back(CopyDesc{PolyRef{R_VAL, pk.slot_lk(l, 0)}, usable, r0, bf + 1});
      cd.push_back(CopyDesc{PolyRef{R_VAL, pk.slot_lk(l, 1)}, usable, r0 + bf + 1, bf + 1});
      reqs.push_back({PolyRef{R_VAL, pk.slot_lk(l, 0)}, true});
      reqs.push_back({PolyRef{R_VAL, pk.slot_lk(l, 1)}, true});
      for (uint32_t b = 0; b < B; ++b) {
        bl[b][2 * l] = rnd_host(ps[b], F, r0 + 2 * (bf + 1));
        bl[b][2 * l + 1] = rnd_host(ps[b], F, r0 + 2 * (bf + 1) + 1);
        ps[b].blinds[G + 3 * l + 0] = bl[b][2 * l]; ps[b].blinds[G + 3 * l + 1] = bl[b][2 * l + 1];
      }
    }
    launch_copy(cd, n);
    commit(reqs, bl, pts);
    for (uint32_t b = 0; b < B; ++b)
      if (w.h_err[b]) throw Error(BZ_ERR_SYNTHESIS, "lookup input not in table (Error::ConstraintSystemFailure) in proof " + std::to_string(b) + " of the batch");
    for (uint32_t b = 0; b < B; ++b) for (uint32_t j = 0; j < 2 * L; ++j) t_write_point(ps[b], pts[b][j]);
  }
  // ---- step 6
  for (uint32_t b = 0; b < B; ++b) {
    HFe beta = t_squeeze(ps[b], F), gamma = t_squeeze(ps[b], F);
    ps[b].consts[pk.C_BETA] = beta; ps[b].consts[pk.C_GAMMA] = gamma;
    HFe bd = beta, delta = F.delta();
    for (uint32_t j = 0; j < pk.M; ++j) { ps[b].consts[pk.C_BD0 + j] = bd; bd = F.mul(bd, delta); }
  }
  upload_consts();
  desc_off = 0;
  // ---- steps 7-9: permutation products, lookup products, random polynomial: one commitment batch
  phase.reset(); phase.reset(new NvtxRange("steps 7-9: grand products, random polynomial"));
  {
    auto perm_desc = [&](uint32_t s) {
      PermSetDesc d{};
      uint32_t c0 = s * pk.chunk_len, c1 = std::min<uint32_t>(pk.M, c0 + pk.chunk_len);
      d.ncols = c1 - c0;
      for (uint32_t j = c0; j < c1; ++j) {
        auto col = cs.perm[j];
        d.val_kind[j - c0] = col.first == 1 ? R_SHVAL : R_VAL;
        d.val_slot[j - c0] = col.first == 0 ? col.second : (col.first == 1 ? col.second : pk.slot_inst(col.second));
        d.sigma_slot[j - c0] = j;
        d.bd_const[j - c0] = pk.C_BD0 + j;
      }
      return d;
    };
    const uint32_t NG = pk.nsets + L;
    const bool gp_sequential = [] { const char* e = getenv("BZ_GP_SEQUENTIAL"); return e && atoi(e) != 0; }();     // A/B knob (read per call)
    if (NG >= 1 && NG <= 8 && (n + SCAN_TILE - 1) / SCAN_TILE <= 8 && !gp_sequential) {
      // Shot / Board: all grand products of the batch in lockstep -- fractions, ONE prefix and ONE suffix scan launch over
      // NG x B arrays, ONE finish launch (a single inversion latency per batch instead of one per product), one copy launch
      const uint64_t PS = (uint64_t)B * n;
      DFe* num = (DFe*)w.nd.p; DFe* den = num + NG * PS; DFe* pnum = den + NG * PS; DFe* sden = pnum + NG * PS;
      GpBatchDesc gd{}; gd.nprod = NG; gd.nsets = pk.nsets;
      std::vector<CopyDesc> cd;
      {
        ProfScope prof(C, PROF_SCAN);
        for (uint32_t s = 0; s < pk.nsets; ++s) {
          perm_fraction_kernel<FpP><<<dim3((n + 127) / 128, B), 128, 0, st>>>(reg, n, perm_desc(s), (const DFe*)pk.lval.p + (uint64_t)cs.F * n, (const DFe*)pk.omega_pows.p,
                                                                            (const DFe*)w.consts.p, pk.cstride, pk.C_BETA, pk.C_GAMMA, num + s * PS, den + s * PS, n);
          gd.zref[s] = PolyRef{R_VAL, pk.slot_pz(s)};
          cd.push_back(CopyDesc{PolyRef{R_VAL, pk.slot_pz(s)}, n - bf, pk.r_perm0 + s * (bf + 1), bf});
        }
        for (uint32_t l = 0; l < L; ++l) {
          const uint32_t g = pk.nsets + l;
          lookup_fraction_kernel<FpP><<<dim3((n + 127) / 128, B), 128, 0, st>>>(reg, n, PolyRef{R_MISC, pk.m_cin0 + 2 * l}, PolyRef{R_MISC, pk.m_cin0 + 2 * l + 1},
                                                                              PolyRef{R_VAL, pk.slot_lk(l, 0)}, PolyRef{R_VAL, pk.slot_lk(l, 1)},
                                                                              (const DFe*)w.consts.p, pk.cstride, pk.C_BETA, pk.C_GAMMA, num + g * PS, den + g * PS, n);
          gd.zref[g] = PolyRef{R_VAL, pk.slot_lk(l, 2)};
          cd.push_back(CopyDesc{PolyRef{R_VAL, pk.slot_lk(l, 2)}, n - bf, pk.r_lkz0 + l * (bf + 1), bf});
        }
        product_scan_kernel<FpP><<<dim3(1, NG * B), SCAN_THREADS, 0, st>>>(num, pnum, n, n, 0);
        product_scan_kernel<FpP><<<dim3(1, NG * B), SCAN_THREADS, 0, st>>>(den, sden, n, n, 1);
        // One CTA per (proof, product), i.e. B x NG inversions per batch instead of one per 128 rows (the r1h launch list shows
        // the 3 072 single-lane chains of the wide geometry costing the fma pipe as much as an IPA-round MSM; r2 A/B on B200:
        // scan scope 5.77 -> 2.78 ms per 5 x 64 proofs, Shot 3 469 -> 3 600 proofs/s).
        grand_product_finish_batch_kernel<FpP><<<dim3(1, B, NG), 256, 0, st>>>(pnum, sden, PS, n, reg, gd, n, n - (bf + 1));
        C->kernel_launches += NG + 3;
      }
      launch_copy(cd, n);
    } else {
    DFe* num = (DFe*)w.nd.p; DFe* den = num + (uint64_t)B * n;
    for (uint32_t s = 0; s < pk.nsets; ++s) {
      PermSetDesc d = perm_desc(s);
      {
        ProfScope prof(C, PROF_SCAN);
        perm_fraction_kernel<FpP><<<dim3((n + 127) / 128, B), 128, 0, st>>>(reg, n, d, (const DFe*)pk.lval.p + (uint64_t)cs.F * n, (const DFe*)pk.omega_pows.p,
                                                                          (const DFe*)w.consts.p, pk.cstride, pk.C_BETA, pk.C_GAMMA, num, den, n);
        C->kernel_launches++;
      }
      grand_product(PolyRef{R_VAL, pk.slot_pz(s)}, s > 0, PolyRef{R_VAL, s > 0 ? pk.slot_pz(s - 1) : 0}, n - (bf + 1));
      std::vector<CopyDesc> cd{CopyDesc{PolyRef{R_VAL, pk.slot_pz(s)}, n - bf, pk.r_perm0 + s * (bf + 1), bf}};
      launch_copy(cd, n);
    }
    for (uint32_t l = 0; l < L; ++l) {
      {
        ProfScope prof(C, PROF_SCAN);
        lookup_fraction_kernel<FpP><<<dim3((n + 127) / 128, B), 128, 0, st>>>(reg, n, PolyRef{R_MISC, pk.m_cin0 + 2 * l}, PolyRef{R_MISC, pk.m_cin0 + 2 * l + 1},
                                                                            PolyRef{R_VAL, pk.slot_lk(l, 0)}, PolyRef{R_VAL, pk.slot_lk(l, 1)},
                                                                            (const DFe*)w.consts.p, pk.cstride, pk.C_BETA, pk.C_GAMMA, num, den, n);
        C->kernel_launches++;
      }
      grand_product(PolyRef{R_VAL, pk.slot_lk(l, 2)}, false, PolyRef{R_VAL, 0}, 0);
      std::vector<CopyDesc> cd{CopyDesc{PolyRef{R_VAL, pk.slot_lk(l, 2)}, n - bf, pk.r_lkz0 + l * (bf + 1), bf}};
      launch_copy(cd, n);
    }
    }
    std::vector<CommitReq> reqs;
    std::vector<std::vector<HFe>> bl(B);
    for (uint32_t s = 0; s < pk.nsets; ++s) reqs.push_back({PolyRef{R_VAL, pk.slot_pz(s)}, true});
    for (uint32_t l = 0; l < L; ++l) reqs.push_back({PolyRef{R_VAL, pk.slot_lk(l, 2)}, true});
    for (uint32_t b = 0; b < B; ++b) {
      for (uint32_t s = 0; s < pk.nsets; ++s) { HFe x = rnd_host(ps[b], F, pk.r_perm0 + s * (bf + 1) + bf); bl[b].push_back(x); ps[b].blinds[G + 3 * L + s] = x; }
      for (uint32_t l = 0; l < L; ++l) { HFe x = rnd_host(ps[b], F, pk.r_lkz0 + l * (bf + 1) + bf); bl[b].push_back(x); ps[b].blinds[G + 3 * l + 2] = x; }
    }
    if (getenv("BZ_SANITY_CHECKS")) {
      // halo2_proofs' `sanity-checks` feature (U: plonk/permutation/prover.rs, plonk/lookup/prover.rs): every grand product
      // must return to 1 on the first unusable row; otherwise the witness violates a copy constraint / lookup
      std::vector<uint32_t> slots;
      if (pk.nsets) slots.push_back(pk.slot_pz(pk.nsets - 1));
      for (uint32_t l = 0; l < L; ++l) slots.push_back(pk.slot_lk(l, 2));
      std::vector<HFe> zs((size_t)B * slots.size());
      for (uint32_t b = 0; b < B; ++b)
        for (size_t j = 0; j < slots.size(); ++j)
          BZ_CUDA(cudaMemcpyAsync(&zs[(size_t)b * slots.size() + j], val(b, slots[j]) + (n - (bf + 1)), 32, cudaMemcpyDeviceToHost, st));
      BZ_CUDA(cudaStreamSynchronize(st));
      for (const HFe& z : zs)
        if (!(z == F.one())) throw Error(BZ_ERR_SYNTHESIS, "sanity check: a grand product does not end in 1 (Error::ConstraintSystemFailure)");
    }
    if (!reqs.empty()) {
      commit(reqs, bl, pts);
      for (uint32_t b = 0; b < B; ++b) for (size_t j = 0; j < reqs.size(); ++j) t_write_point(ps[b], pts[b][j]);
    }
    // random polynomial (coefficient basis g)
    std::vector<CommitReq> rq{{PolyRef{R_RANDPOLY, 0}, false}};
    std::vector<std::vector<HFe>> rb(B, std::vector<HFe>(1));
    for (uint32_t b = 0; b < B; ++b) { rb[b][0] = rnd_host(ps[b], F, pk.r_rand_blind); ps[b].blinds[pk.nblinds - 1] = rb[b][0]; }
    commit(rq, rb, pts);
    for (uint32_t b = 0; b < B; ++b) t_write_point(ps[b], pts[b][0]);
    // polys + cosets of lookup columns and z's
    to_coeff(G + I, 3 * L + pk.nsets);
    to_coset(G + I, 3 * L + pk.nsets);
  }
  // ---- step 10
  for (uint32_t b = 0; b < B; ++b) {
    const HFe y = t_squeeze(ps[b], F);
    ps[b].consts[pk.C_Y] = y;
    HFe yp = F.one();
    for (uint32_t g = 0; g <= pk.n_exprs; ++g) { ps[b].consts[pk.C_YP0 + g] = yp; yp = F.mul(yp, y); }
  }
  upload_consts();
  desc_off = 0;
  // ---- steps 11-12: h(X)
  phase.reset(); phase.reset(new NvtxRange("steps 11-13: h(X), pieces"));
  {
    compute_h();
    std::vector<CommitReq> reqs;
    std::vector<std::vector<HFe>> bl(B, std::vector<HFe>(pk.qdeg));
    for (uint32_t i = 0; i < pk.qdeg; ++i) reqs.push_back({PolyRef{R_HCOEF, i}, false});
    for (uint32_t b = 0; b < B; ++b) for (uint32_t i = 0; i < pk.qdeg; ++i) bl[b][i] = rnd_host(ps[b], F, pk.r_hblind + i);
    commit(reqs, bl, pts);
    for (uint32_t b = 0; b < B; ++b) for (uint32_t i = 0; i < pk.qdeg; ++i) t_write_point(ps[b], pts[b][i]);
    // ---- step 13: x
    for (uint32_t b = 0; b < B; ++b) {
      HFe x = t_squeeze(ps[b], F);
      ps[b].consts[pk.C_X] = x;
      HFe xn = x; for (uint32_t i = 0; i < k; ++i) xn = F.sqr(xn);
      ps[b].consts[pk.C_XN] = xn;
      for (int r : pk.rots) {
        HFe pt = r >= 0 ? F.mul(x, F.pow_u64(pk.omega, (uint64_t)r)) : F.mul(x, F.pow_u64(pk.omega_inv, (uint64_t)(-r)));
        ps[b].consts[pk.rot_const.at(r)] = pt;
      }
      // h blind: fold from the last piece
      HFe hb = F.zero();
      for (int i = (int)pk.qdeg - 1; i >= 0; --i) hb = F.add(F.mul(hb, xn), bl[b][i]);
      ps[b].blinds[pk.nblinds - 2] = hb;
    }
    upload_consts();
    // h_poly = sum pieces_i xn^i (Horner from the last piece)
    std::vector<PolyRef> refs;
    for (int i = (int)pk.qdeg - 1; i >= 0; --i) refs.push_back(PolyRef{R_HCOEF, (uint32_t)i});
    std::vector<LinCombDesc> ld{LinCombDesc{PolyRef{R_MISC, pk.m_hpoly}, pk.C_XN, pk.qdeg, 0}};
    lincomb(ld, refs);
  }
  // ---- steps 14-18: evaluations
  phase.reset(); phase.reset(new NvtxRange("steps 14-18: evaluations"));
  {
    std::vector<std::vector<HFe>> ev;
    evaluate((const EvalQuery*)pk.d_evals.p, (uint32_t)pk.evals.size(), ev);
    for (uint32_t b = 0; b < B; ++b) for (const HFe& e : ev[b]) t_write_scalar(ps[b], F, e);
  }
  // ---- step 20: multiopen
  phase.reset(); phase.reset(new NvtxRange("step 20: multiopen"));
  const uint32_t nps = (uint32_t)pk.point_sets.size();
  std::vector<std::vector<HFe>> q_blinds(B, std::vector<HFe>(nps));
  {
    for (uint32_t b = 0; b < B; ++b) { ps[b].consts[pk.C_X1] = t_squeeze(ps[b], F); ps[b].consts[pk.C_X2] = t_squeeze(ps[b], F); }
    upload_consts();
    desc_off = 0;
    std::vector<LinCombDesc> ld;
    std::vector<PolyRef> refs;
    for (uint32_t s = 0; s < nps; ++s) {
      uint32_t first = (uint32_t)refs.size(), cnt = 0;
      for (auto& ci : pk.cmap) if (ci.set == (int)s) { refs.push_back(ci.poly); ++cnt; }
      ld.push_back(LinCombDesc{PolyRef{R_MISC, pk.m_qset0 + s}, pk.C_X1, cnt, first});
    }
    lincomb(ld, refs);
    for (uint32_t b = 0; b < B; ++b) {
      const HFe x1 = ps[b].consts[pk.C_X1];
      for (uint32_t s = 0; s < nps; ++s) q_blinds[b][s] = F.zero();
      for (auto& ci : pk.cmap) {
        HFe bl = ci.blind_kind == 0 ? F.one() : ps[b].blinds[ci.blind_idx];
        q_blinds[b][ci.set] = F.add(F.mul(q_blinds[b][ci.set], x1), bl);
      }
    }
    // successive synthetic divisions; round r divides every set that has > r points
    size_t maxpts = 0;
    for (auto& s : pk.point_sets) maxpts = std::max(maxpts, s.size());
    std::vector<PolyRef> cur(nps);
    for (uint32_t s = 0; s < nps; ++s) cur[s] = PolyRef{R_MISC, pk.m_qset0 + s};
    for (size_t r = 0; r < maxpts; ++r) {
      std::vector<KateDesc> kd;
      for (uint32_t s = 0; s < nps; ++s)
        if (pk.point_sets[s].size() > r) {
          PolyRef outp{R_MISC, pk.m_qtmp0 + 2 * s + (uint32_t)(r & 1)};
          kd.push_back(KateDesc{cur[s], outp, pk.rot_const.at(pk.point_sets[s][r])});
          cur[s] = outp;
        }
      KateDesc* dk = upload_desc(kd);
      ProfScope prof(C, PROF_POLY);
      const uint32_t splits = std::max(1u, n / 16384u);
      if (splits == 1) kate_division_kernel<FpP><<<dim3((unsigned)kd.size(), B), KATE_THREADS, 0, st>>>(reg, n, dk, (const DFe*)w.consts.p, pk.cstride);
      else {                       // large domains: slice totals, chain, redo with the carry-in
        const size_t slots = (size_t)B * kd.size() * splits;
        w.eval_tmp.ensure(2 * slots * 32);
        DFe* totals = (DFe*)w.eval_tmp.p; DFe* carries = totals + slots;
        kate_division_kernel<FpP><<<dim3((unsigned)kd.size(), B, splits), KATE_THREADS, 0, st>>>(reg, n, dk, (const DFe*)w.consts.p, pk.cstride, nullptr, totals);
        kate_carry_kernel<FpP><<<(unsigned)((B * kd.size() + 63) / 64), 64, 0, st>>>(n, splits, (uint32_t)kd.size(), B, dk, (const DFe*)w.consts.p, pk.cstride, totals, carries);
        kate_division_kernel<FpP><<<dim3((unsigned)kd.size(), B, splits), KATE_THREADS, 0, st>>>(reg, n, dk, (const DFe*)w.consts.p, pk.cstride, carries, nullptr);
        C->kernel_launches += 2;
      }
      C->kernel_launches++;
    }
    std::vector<LinCombDesc> l2{LinCombDesc{PolyRef{R_MISC, pk.m_qprime}, pk.C_X2, nps, 0}};
    lincomb(l2, cur);
    std::vector<CommitReq> rq{{PolyRef{R_MISC, pk.m_qprime}, false}};
    std::vector<std::vector<HFe>> qb(B, std::vector<HFe>(1));
    for (uint32_t b = 0; b < B; ++b) qb[b][0] = rnd_host(ps[b], F, pk.r_qprime);
    commit(rq, qb, pts);
    for (uint32_t b = 0; b < B; ++b) t_write_point(ps[b], pts[b][0]);
    for (uint32_t b = 0; b < B; ++b) ps[b].consts[pk.C_X3] = t_squeeze(ps[b], F);
    upload_consts();
    std::vector<EvalQuery> eq;
    for (uint32_t s = 0; s < nps; ++s) eq.push_back(EvalQuery{PolyRef{R_MISC, pk.m_qset0 + s}, pk.C_X3});
    EvalQuery* deq = upload_desc(eq);
    std::vector<std::vector<HFe>> ev;
    evaluate(deq, nps, ev);
    for (uint32_t b = 0; b < B; ++b) for (const HFe& e : ev[b]) t_write_scalar(ps[b], F, e);
    for (uint32_t b = 0; b < B; ++b) ps[b].consts[pk.C_X4] = t_squeeze(ps[b], F);
    upload_consts();
    std::vector<PolyRef> prefs{PolyRef{R_MISC, pk.m_qprime}};
    for (uint32_t s = 0; s < nps; ++s) prefs.push_back(PolyRef{R_MISC, pk.m_qset0 + s});
    std::vector<LinCombDesc> l3{LinCombDesc{PolyRef{R_MISC, pk.m_ppoly}, pk.C_X4, nps + 1, 0}};
    lincomb(l3, prefs);
    for (uint32_t b = 0; b < B; ++b) {
      HFe pb = qb[b][0], x4 = ps[b].consts[pk.C_X4];
      for (uint32_t s = 0; s < nps; ++s) pb = F.add(F.mul(pb, x4), q_blinds[b][s]);
      q_blinds[b].push_back(pb);        // stash p_blind at index nps
    }
  }
  // ---- step 21: inner product argument
  phase.reset(); phase.reset(new NvtxRange("step 21: inner product argument"));
  {
    desc_off = 0;
    // S(X): random coefficients with S(x3) = 0
    std::vector<EvalQuery> eq{EvalQuery{PolyRef{R_SPOLY, 0}, pk.C_X3}};
    EvalQuery* deq = upload_desc(eq);
    {
      ProfScope prof(C, PROF_EVAL);
      eval_launch(deq, 1);
      tweak_element_kernel<FpP><<<(B + 63) / 64, 64, 0, st>>>(reg, n, PolyRef{R_SPOLY, 0}, 0, (const DFe*)w.evalout.p, 1, 0, 0, B);
      C->kernel_launches += 1;
    }
    std::vector<CommitReq> rq{{PolyRef{R_SPOLY, 0}, false}};
    std::vector<std::vector<HFe>> sb(B, std::vector<HFe>(1));
    for (uint32_t b = 0; b < B; ++b) sb[b][0] = rnd_host(ps[b], F, pk.r_sblind);
    commit(rq, sb, pts);
    std::vector<HFe> fblind(B);
    for (uint32_t b = 0; b < B; ++b) {
      t_write_point(ps[b], pts[b][0]);
      HFe xi = t_squeeze(ps[b], F), z = t_squeeze(ps[b], F);
      ps[b].consts[pk.C_XI] = xi; ps[b].consts[pk.C_Z] = z;
      fblind[b] = F.add(F.mul(sb[b][0], xi), q_blinds[b][nps]);
    }
    upload_consts();
    // p' = S * xi + P ; p'[0] -= p'(x3) ; b = powers of x3 ; coef = 1
    std::vector<PolyRef> refs{PolyRef{R_SPOLY, 0}, PolyRef{R_MISC, pk.m_ppoly}};
    std::vector<LinCombDesc> ld{LinCombDesc{PolyRef{R_MISC, pk.m_pprime}, pk.C_XI, 2, 0}};
    lincomb(ld, refs);
    std::vector<EvalQuery> eq2{EvalQuery{PolyRef{R_MISC, pk.m_pprime}, pk.C_X3}};
    EvalQuery* deq2 = upload_desc(eq2);
    {
      ProfScope prof(C, PROF_IPA);
      eval_launch(deq2, 1);
      tweak_element_kernel<FpP><<<(B + 63) / 64, 64, 0, st>>>(reg, n, PolyRef{R_MISC, pk.m_pprime}, 0, (const DFe*)w.evalout.p, 1, 0, 0, B);
      powers_kernel<FpP><<<dim3((n + 127) / 128, B), 128, 0, st>>>(reg, n, PolyRef{R_MISC, pk.m_b}, (const DFe*)w.consts.p, pk.cstride, pk.C_X3);
      fill_kernel<FpP><<<dim3((n + 127) / 128, B), 128, 0, st>>>(reg, n, PolyRef{R_MISC, pk.m_coef}, n, dfe(F.one()));
      C->kernel_launches += 3;
    }
    // rounds
    std::vector<void*> mainp((size_t)B * 2), extrap((size_t)B * 2);
    for (uint32_t b = 0; b < B; ++b) {
      mainp[2 * b] = misc(b, pk.m_scl); mainp[2 * b + 1] = misc(b, pk.m_scr);
      extrap[2 * b] = (DFe*)w.extras.p + (size_t)b * 4; extrap[2 * b + 1] = (DFe*)w.extras.p + (size_t)b * 4 + 2;
    }
    const uint32_t n_msm = 2 * B;
    pts.assign(B, std::vector<HostPoint>(2));
    // Late rounds of one LARGE proof.  L_j / R_j are MSMs over the ORIGINAL g with the scalars p'[i' ^ half] * coef[o], n points
    // in every round however short p' has become (no generator folding, DESIGN.md section 3).  Once G'_j is down to len0 = 2^mat_log
    // points it is materialised instead:  G'[i'] = sum_q coef[q * len0 + i'] * g[q * len0 + i'],  where coef depends on q only (the
    // challenges so far act on the high index bits) -- len0 MSMs that share ONE scalar vector (msm_multi_run: one sort, coalesced
    // base loads, the cost of about one round) -- and the remaining rounds are the same algorithm on len0 points (coef := 1).
    // k = 20: 10 of the 20 rounds shrink from n to 1024 points (proof 335 -> 290 ms; k = 18: 100 -> 83 ms; at k = 16 a table-MSM
    // round is already cheaper than the fixed latency of a small bucket MSM: 26 -> 32 ms, so the default starts at k = 18).  Batch
    // of one only (G' differs per proof); BZ_IPA_MATERIALIZE_LOG picks log2(len0) (0 = off).
    uint32_t mat_log = (B == 1 && k >= 18) ? 10u : 0u;
    if (const char* e = getenv("BZ_IPA_MATERIALIZE_LOG")) mat_log = (B == 1) ? (uint32_t)atoi(e) : 0u;
    if (mat_log < 2 || mat_log + 1 > k || (n >> mat_log) > 4096) mat_log = 0;
    const uint32_t len0 = mat_log ? (1u << mat_log) : 0, j_mat = mat_log ? k - mat_log : k;
    uint32_t count = n;                       // length of the generator vector the scalars of the current round refer to
    const int curve = pk.params->curve;
    for (uint32_t j = 0; j < k; ++j) {
      const uint32_t half = 1u << (k - j - 1);
      if (mat_log && j == j_mat) {
        ProfScope prof(C, PROF_IPA);
        const uint32_t nq = n >> mat_log;
        w.ipa_coefq.ensure((size_t)nq * 32); w.ipa_gm.ensure(((size_t)len0 + 2) * 64); w.msm_jac.ensure((size_t)len0 * 96);
        BZ_CUDA(cudaMemcpy2DAsync(w.ipa_coefq.p, 32, misc(0, pk.m_coef), (size_t)len0 * 32, 32, nq, cudaMemcpyDeviceToDevice, st));
        msm_multi_run(C, curve, w.ipa_coefq.p, nq, pk.params->g_w_u.p, len0, len0, w.msm_jac.p);
        jac_to_affine_run(C, curve, w.msm_jac.p, w.ipa_gm.p, len0);
        BZ_CUDA(cudaMemcpyAsync((char*)w.ipa_gm.p + (size_t)len0 * 64, (const char*)pk.params->g_w_u.p + (size_t)n * 64, 128, cudaMemcpyDeviceToDevice, st));   // w, u
        fill_kernel<FpP><<<dim3((len0 + 127) / 128, B), 128, 0, st>>>(reg, n, PolyRef{R_MISC, pk.m_coef}, len0, dfe(F.one()));
        C->kernel_launches++;
        count = len0;
      }
      {
        ProfScope prof(C, PROF_IPA);
        ipa_scalars_kernel<FpP><<<dim3((count + 127) / 128, B), 128, 0, st>>>(reg, n, count, half, PolyRef{R_MISC, pk.m_pprime}, PolyRef{R_MISC, pk.m_coef},
                                                                            PolyRef{R_MISC, pk.m_scl}, PolyRef{R_MISC, pk.m_scr});
        if (half >= (1u << 15)) {
          // long vectors: a single CTA per proof took 0.4 ms per round at k = 20 (3 % of the proof); slices across the GPU instead
          const uint32_t parts = std::min<uint32_t>(128, half >> 12);
          w.ipa_tmp.ensure((size_t)B * parts * 2 * 32);
          ipa_inner_partial_kernel<FpP><<<dim3(B, parts), IPA_THREADS, 0, st>>>(reg, n, half, PolyRef{R_MISC, pk.m_pprime}, PolyRef{R_MISC, pk.m_b}, (DFe*)w.ipa_tmp.p);
          ipa_inner_finish_kernel<FpP><<<B, 128, 0, st>>>((const DFe*)w.ipa_tmp.p, parts, (const DFe*)w.consts.p, pk.cstride, pk.C_Z, (const DFe*)w.rnd.p, pk.R,
                                                         pk.r_ipa + 2 * j, pk.r_ipa + 2 * j + 1, (DFe*)w.extras.p);
          C->kernel_launches++;
        } else
        ipa_inner_kernel<FpP><<<B, IPA_THREADS, 0, st>>>(reg, n, half, PolyRef{R_MISC, pk.m_pprime}, PolyRef{R_MISC, pk.m_b}, (const DFe*)w.consts.p, pk.cstride,
                                                        pk.C_Z, (const DFe*)w.rnd.p, pk.R, pk.r_ipa + 2 * j, pk.r_ipa + 2 * j + 1, (DFe*)w.extras.p);
        C->kernel_launches += 2;
      }
      if (count == n) {
        run_msms(false, mainp, extrap, n_msm);
        read_points(n_msm, 2, pts);
      } else {
        // bucket MSM of the two short vectors over G' || w || u; every rank of a sharded proof computes it (it is tiny)
        const void* const* dm = upload_msm_ptrs(C, w.ptrs, mainp, extrap);
        w.msm_jac.ensure((size_t)n_msm * 96);
        msm_run_batch(C, curve, dm, dm + n_msm, count, 0, count + 2, w.ipa_gm.p, n_msm, w.msm_jac.p);
        jac_to_affine_run(C, curve, w.msm_jac.p, w.commits.p, n_msm);
        read_points(n_msm, 2, pts, true);
      }
      std::vector<HFe> us(B), uinvs(B);
      for (uint32_t b = 0; b < B; ++b) {
        t_write_point(ps[b], pts[b][0]);
        t_write_point(ps[b], pts[b][1]);
        us[b] = t_squeeze(ps[b], F);
      }
      uinvs = us;
      host_batch_invert(F, uinvs);                  // one inversion per round for the whole batch
      for (uint32_t b = 0; b < B; ++b) {
        const HFe u = us[b], uinv = uinvs[b];
        ps[b].consts[pk.C_U] = u; ps[b].consts[pk.C_UINV] = uinv;
        HFe lr = rnd_host(ps[b], F, pk.r_ipa + 2 * j), rr = rnd_host(ps[b], F, pk.r_ipa + 2 * j + 1);
        fblind[b] = F.add(fblind[b], F.add(F.mul(lr, uinv), F.mul(rr, u)));
      }
      upload_consts();
      ProfScope prof(C, PROF_IPA);
      ipa_fold_kernel<FpP><<<dim3((count + 127) / 128, B), 128, 0, st>>>(reg, n, count, half, PolyRef{R_MISC, pk.m_pprime}, PolyRef{R_MISC, pk.m_b}, PolyRef{R_MISC, pk.m_coef},
                                                                   (const DFe*)w.consts.p, pk.cstride, pk.C_U, pk.C_UINV);
      C->kernel_launches++;
    }
    // c = p'[0], f
    for (uint32_t b = 0; b < B; ++b) BZ_CUDA(cudaMemcpyAsync((char*)w.h_pinned + (size_t)b * 32, misc(b, pk.m_pprime), 32, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
    for (uint32_t b = 0; b < B; ++b) {
      HFe c; memcpy(c.l, (char*)w.h_pinned + (size_t)b * 32, 32);
      t_write_scalar(ps[b], F, c);
      t_write_scalar(ps[b], F, fblind[b]);
      BZ_CHECK(ps[b].pos == pk.proof_size, "internal: proof size mismatch");
    }
  }
  BZ_CUDA(cudaGetLastError());
}

}  // namespace bz

extern "C" API int bz_create_proofs(bz_ctx* ctx, bz_pk* pkh, uint32_t batch, const void* instances, const uint32_t* instance_lens,
                                    uint32_t instance_stride, const void* advice, const void* rand_wide, void* proofs) {
  PV_TRY(ctx, {
    BZ_CHECK(pkh && advice && rand_wide && proofs && batch >= 1, "null argument");
    PkImpl& pk = pkh->p;
    BZ_CHECK(pk.cs.I == 0 || (instances && instance_lens), "instances missing");
    ensure_work(C, pk, batch);
    Prover pr(C, pk, batch);
    pr.run(instances, instance_lens, instance_stride, advice, rand_wide, (uint8_t*)proofs);
  });
}

// The same proofs with the blinding randomness expanded on the device: proof b is bz_create_proofs' proof with rand_wide[b] =
// the ChaCha20 keystream of seeds[b].  The stream is written into the staging buffer bz_create_proofs copies rand_wide to, and
// Prover::run takes it from there through its device-pointer path (the short ranges the host reads are mirrored back).
extern "C" API int bz_create_proofs_seeded(bz_ctx* ctx, bz_pk* pkh, uint32_t batch, const void* instances, const uint32_t* instance_lens,
                                           uint32_t instance_stride, const void* advice, const void* seeds, void* proofs) {
  PV_TRY(ctx, {
    BZ_CHECK(pkh && advice && seeds && proofs && batch >= 1, "null argument");
    PkImpl& pk = pkh->p;
    BZ_CHECK(pk.cs.I == 0 || (instances && instance_lens), "instances missing");
    // the same seed for two witnesses would give both proofs the same blinds, which breaks zero knowledge
    std::set<std::array<uint8_t, 32>> distinct;
    for (uint32_t b = 0; b < batch; ++b) {
      std::array<uint8_t, 32> s;
      memcpy(s.data(), (const uint8_t*)seeds + (size_t)b * 32, 32);
      BZ_CHECK(distinct.insert(s).second, "bz_create_proofs_seeded: seed " + std::to_string(b) + " repeats an earlier seed of the batch");
    }
    ensure_work(C, pk, batch);
    PkImpl::Work& w = pk.work;
    w.seeds.ensure((size_t)batch * 32);
    BZ_CUDA(cudaMemcpyAsync(w.seeds.p, seeds, (size_t)batch * 32, cudaMemcpyHostToDevice, C->stream));
    chacha20_fill_run(C, w.seeds.p, batch, pk.R, w.wide.p);
    Prover pr(C, pk, batch);
    pr.run(instances, instance_lens, instance_stride, advice, w.wide.p, (uint8_t*)proofs);
  });
}

// ======================================================================================================
// Fine-grained entry points bound to a ProvingKey / Params (SURVEY 8b minimum export set): what a patched
// plonk/vanishing/prover.rs and poly/commitment/prover.rs would call one-for-one.  Host buffers, synchronous.
// ======================================================================================================
extern "C" {

// vanishing::Argument::construct up to h(X)'s coefficients (U: halo2_proofs 0.2.0 src/plonk/vanishing/prover.rs `construct`,
// src/plonk/prover.rs the `h_poly` expression list, src/poly/domain.rs `divide_by_vanishing_poly` + `extended_to_coeff`).
API int bz_pk_quotient(bz_ctx* ctx, bz_pk* pkh, const void* polys, const void* theta, const void* beta, const void* gamma, const void* y, void* out_h) {
  if (!ctx) return BZ_ERR_INVALID;
  PV_TRY(ctx, {
    BZ_CHECK(pkh && polys && theta && beta && gamma && y && out_h, "null argument");
    PkImpl& pk = pkh->p;
    ensure_work(C, pk, 1);
    Prover pr(C, pk, 1);
    const bzh::Field& F = C->fp;
    ProofState& ps = pr.ps[0];
    ps.consts.assign(pk.cstride, F.zero());
    for (uint32_t i = 0; i < pk.NC; ++i) ps.consts[i] = pk.cs.consts[i];
    ps.consts[pk.C_ONE] = F.one();
    HFe th, be, ga, yy;
    memcpy(th.l, theta, 32); memcpy(be.l, beta, 32); memcpy(ga.l, gamma, 32); memcpy(yy.l, y, 32);
    ps.consts[pk.C_THETA] = th; ps.consts[pk.C_BETA] = be; ps.consts[pk.C_GAMMA] = ga; ps.consts[pk.C_Y] = yy;
    HFe bd = be;
    for (uint32_t j = 0; j < pk.M; ++j) { ps.consts[pk.C_BD0 + j] = bd; bd = F.mul(bd, F.delta()); }
    HFe yp = F.one();
    for (uint32_t g = 0; g <= pk.n_exprs; ++g) { ps.consts[pk.C_YP0 + g] = yp; yp = F.mul(yp, yy); }
    pr.upload_consts();
    BZ_CUDA(cudaMemcpyAsync(pr.w.poly.p, polys, (size_t)pk.NS * pk.n * 32, cudaMemcpyHostToDevice, pr.st));
    pr.to_coset(0, pk.NS);
    pr.compute_h();
    BZ_CUDA(cudaMemcpyAsync(out_h, pr.w.hcoef.p, (size_t)pk.qdeg * pk.n * 32, cudaMemcpyDeviceToHost, pr.st));
    BZ_CUDA(cudaStreamSynchronize(pr.st));
  });
}
API uint32_t bz_pk_num_poly_slots(const bz_pk* pk) { return pk ? pk->p.NS : 0; }

}  // extern "C"

// ---- inner product argument, round by round (U: halo2_proofs 0.2.0 src/poly/commitment/prover.rs `create_proof`) ----
struct bz_ipa {
  bz::ParamsImpl* params = nullptr;
  uint32_t n = 0, k = 0, round = 0;
  bz::DevBuf vec;        // 5 x n scalars: p', b, coef (challenge products over the ORIGINAL g), scalars of L, scalars of R
  bz::DevBuf consts;     // z, u, u^-1, x3
  bz::DevBuf rnd;        // l_rand, r_rand
  bz::DevBuf extras;     // [2][2] extra scalars of the two MSMs (w: blind, u: z <p', b>)
  bz::DevBuf ptrs, out;
  bz::Regions reg;
};

extern "C" {

API int bz_ipa_begin(bz_ctx* ctx, bz_params* params, const void* p_prime, const void* x3, bz_ipa** out) {
  if (!ctx) return BZ_ERR_INVALID;
  PV_TRY(ctx, {
    BZ_CHECK(params && p_prime && x3 && out, "null argument");
    *out = nullptr;
    std::unique_ptr<bz_ipa> h(new bz_ipa());
    h->params = &params->p; h->n = params->p.n; h->k = params->p.k;
    BZ_CHECK(params->p.curve == 0, "ipa: only the Vesta commitment curve is wired up");
    const size_t n = h->n;
    cudaStream_t st = C->stream;
    h->vec.alloc(5 * n * 32); h->consts.alloc(8 * 32); h->rnd.alloc(2 * 32); h->extras.alloc(4 * 32); h->ptrs.alloc(4 * sizeof(void*)); h->out.alloc(2 * 128);
    memset(&h->reg, 0, sizeof(h->reg));
    h->reg.base[R_MISC] = h->vec.p; h->reg.stride[R_MISC] = 0;
    BZ_CUDA(cudaMemcpyAsync(h->vec.p, p_prime, n * 32, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaMemsetAsync(h->consts.p, 0, 8 * 32, st));
    BZ_CUDA(cudaMemcpyAsync((DFe*)h->consts.p + 3, x3, 32, cudaMemcpyHostToDevice, st));
    powers_kernel<FpP><<<dim3((unsigned)((n + 127) / 128), 1), 128, 0, st>>>(h->reg, (uint32_t)n, PolyRef{R_MISC, 1}, (const DFe*)h->consts.p, 8, 3);
    fill_kernel<FpP><<<dim3((unsigned)((n + 127) / 128), 1), 128, 0, st>>>(h->reg, n, PolyRef{R_MISC, 2}, (uint32_t)n, dfe(C->fp.one()));
    C->kernel_launches += 2;
    void* ptrs[4] = {(DFe*)h->vec.p + 3 * n, (DFe*)h->vec.p + 4 * n, (DFe*)h->extras.p, (DFe*)h->extras.p + 2};
    BZ_CUDA(cudaMemcpyAsync(h->ptrs.p, ptrs, sizeof(ptrs), cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaStreamSynchronize(st));
    *out = h.release();
  });
}

// L_j and R_j of the current round (affine, 64 B each): <p'_hi, G'_lo> + [z <p'_hi, b_lo>] U + [l_rand] W and the mirror image
API int bz_ipa_round(bz_ctx* ctx, bz_ipa* ipa, const void* z, const void* l_rand, const void* r_rand, void* out_l_affine, void* out_r_affine) {
  if (!ctx) return BZ_ERR_INVALID;
  PV_TRY(ctx, {
    BZ_CHECK(ipa && z && l_rand && r_rand && out_l_affine && out_r_affine, "null argument");
    BZ_CHECK(ipa->round < ipa->k, "ipa: all rounds done");
    cudaStream_t st = C->stream;
    const uint32_t n = ipa->n, half = 1u << (ipa->k - ipa->round - 1);
    BZ_CUDA(cudaMemcpyAsync(ipa->consts.p, z, 32, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaMemcpyAsync(ipa->rnd.p, l_rand, 32, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaMemcpyAsync((DFe*)ipa->rnd.p + 1, r_rand, 32, cudaMemcpyHostToDevice, st));
    ipa_scalars_kernel<FpP><<<dim3((n + 127) / 128, 1), 128, 0, st>>>(ipa->reg, n, n, half, PolyRef{R_MISC, 0}, PolyRef{R_MISC, 2}, PolyRef{R_MISC, 3}, PolyRef{R_MISC, 4});
    ipa_inner_kernel<FpP><<<1, IPA_THREADS, 0, st>>>(ipa->reg, n, half, PolyRef{R_MISC, 0}, PolyRef{R_MISC, 1}, (const DFe*)ipa->consts.p, 8, 0,
                                                    (const DFe*)ipa->rnd.p, 0, 0, 1, (DFe*)ipa->extras.p);
    C->kernel_launches += 2;
    // extras are [blind (w), z <p', b> (u)] in the order of g || w || u
    params_commit_run(C, *ipa->params, false, (const void* const*)ipa->ptrs.p, (const void* const*)ipa->ptrs.p + 2, 2, ipa->out.p);
    BZ_CUDA(cudaMemcpyAsync(out_l_affine, ipa->out.p, 64, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaMemcpyAsync(out_r_affine, (char*)ipa->out.p + 64, 64, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}

// p'_lo += u^-1 p'_hi, b_lo += u b_hi, G'_lo += [u] G'_hi (kept as challenge products over the original generators)
API int bz_ipa_fold(bz_ctx* ctx, bz_ipa* ipa, const void* u, const void* u_inv) {
  if (!ctx) return BZ_ERR_INVALID;
  PV_TRY(ctx, {
    BZ_CHECK(ipa && u && u_inv, "null argument");
    BZ_CHECK(ipa->round < ipa->k, "ipa: all rounds done");
    cudaStream_t st = C->stream;
    const uint32_t n = ipa->n, half = 1u << (ipa->k - ipa->round - 1);
    BZ_CUDA(cudaMemcpyAsync((DFe*)ipa->consts.p + 1, u, 32, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaMemcpyAsync((DFe*)ipa->consts.p + 2, u_inv, 32, cudaMemcpyHostToDevice, st));
    ipa_fold_kernel<FpP><<<dim3((n + 127) / 128, 1), 128, 0, st>>>(ipa->reg, n, n, half, PolyRef{R_MISC, 0}, PolyRef{R_MISC, 1}, PolyRef{R_MISC, 2}, (const DFe*)ipa->consts.p, 8, 1, 2);
    C->kernel_launches++;
    BZ_CUDA(cudaStreamSynchronize(st));
    ipa->round++;
  });
}

// c = p'[0] after the last round; releases the state
API int bz_ipa_finish(bz_ctx* ctx, bz_ipa* ipa, void* out_c) {
  if (!ctx) return BZ_ERR_INVALID;
  PV_TRY(ctx, {
    BZ_CHECK(ipa && out_c, "null argument");
    std::unique_ptr<bz_ipa> own(ipa);
    BZ_CHECK(ipa->round == ipa->k, "ipa: rounds missing");
    BZ_CUDA(cudaMemcpyAsync(out_c, ipa->vec.p, 32, cudaMemcpyDeviceToHost, C->stream));
    BZ_CUDA(cudaStreamSynchronize(C->stream));
  });
}
API void bz_ipa_destroy(bz_ipa* ipa) { delete ipa; }

}  // extern "C"


// ---- build-time access to the compiled h(X) programs (no GPU needed): scripts/gen_quotient_kernels.py ------------------------
extern "C" {
API int bz_quotient_program(const bz_circuit* cs, uint32_t tier, uint32_t* code, uint32_t code_cap, uint32_t* n_code, int32_t* rot, uint32_t rot_cap,
                            uint32_t* n_rot, uint64_t* hash) {
  try {
    if (!cs || tier >= PkImpl::Q_TIERS || !n_code || !n_rot) return BZ_ERR_INVALID;
    bzh::Field F{0};
    PkImpl pk;
    pk_host_setup(F, pk, cs);
    const std::vector<uint32_t>& c = pk.h_q_code[tier];
    const std::vector<int32_t>& r = pk.h_q_rot[tier];
    *n_code = (uint32_t)c.size(); *n_rot = (uint32_t)r.size();
    if (hash) *hash = program_hash(c, r);
    if (code && code_cap >= c.size() && !c.empty()) memcpy(code, c.data(), c.size() * 4);
    if (rot && rot_cap >= r.size() && !r.empty()) memcpy(rot, r.data(), r.size() * 4);
    return BZ_OK;
  } catch (const std::exception&) { return BZ_ERR_INVALID; }
}
/* 1 when tier `tier` of this proving key runs circuit-specialised generated code, 0 for the interpreter */
API int bz_pk_quotient_generated(const bz_pk* pk, uint32_t tier) { return pk && tier < PkImpl::Q_TIERS && pk->p.q_gen[tier] ? 1 : 0; }
}
