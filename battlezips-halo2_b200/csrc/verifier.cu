#include "prover_impl.h"

using namespace bz;

// ======================================================================================================
// verify_proof on the device, batch-major (SURVEY §8f rank 4).
// Mirrors halo2_proofs 0.2.0 `plonk::verify_proof` with a SingleVerifier strategy and the verifiers it drives
// (U: src/plonk/verifier.rs, src/plonk/{permutation,lookup,vanishing}/verifier.rs, src/poly/multiopen/verifier.rs,
//  src/poly/commitment/verifier.rs, src/poly/commitment/msm.rs; reference call sites /root/reference/benches/board.rs:84,
//  src/circuits/shot.rs:933-940, src/circuits/board.rs:925-932).
// Host: transcript, challenges, the expected h(x) from the gate expressions, multiopen / IPA scalar bookkeeping (what
// stays Rust in the drop-in).  Device: point decompression (square roots), the instance commitments, compute_s, and the
// whole final check  sum_i a_i P_i + <s, G> + [..]W + [..]U == 0  as one fixed-base table MSM plus one scalar
// multiplication per proof point -- every proof of the batch gets its own verdict.
// ======================================================================================================
namespace bz {

typedef ::bz::Fe<FqP> DFq;

// (point decompression: decompress_points_run in params.cu)

// compute_s (U: poly/commitment/verifier.rs): s[idx] = init * prod_{bit i of idx set} u_rev[i];  s[0] += add0.
// consts per proof: [0] init (= -c), [1] add0 (= -v, the g[0] term), [2 .. 2+k) u_rev
__global__ void compute_s_kernel(const DFe* __restrict__ consts, uint32_t cstride, DFe* __restrict__ s, uint32_t k) {
  const uint32_t n = 1u << k, idx = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (idx >= n) return;
  const DFe* c = consts + (size_t)b * cstride;
  DFe v = fe_load(c);
  for (uint32_t i = 0; i < k; ++i)
    if ((idx >> i) & 1) v = fe_mul(v, fe_load(c + 2 + i));
  if (idx == 0) v = fe_add(v, fe_load(c + 1));
  fe_store(s + (size_t)b * n + idx, v);
}

// one CTA per proof: thread i < nv computes [a_i] P_i (a_i canonical), the CTA sums them, adds the fixed-base part and
// reports whether the total is the identity
constexpr int VFY_THREADS = 128;
__global__ void __launch_bounds__(VFY_THREADS) verify_final_kernel(const Affine<FqP>* __restrict__ pts, const uint32_t* __restrict__ scalars /* nv x 8, canonical */,
                                                                  uint32_t nv, const Affine<FqP>* __restrict__ fixed_part, uint8_t* __restrict__ ok) {
  __shared__ Xyzz<FqP> sh[VFY_THREADS];
  const uint32_t b = blockIdx.x, tid = threadIdx.x;
  Xyzz<FqP> acc = xyzz_identity<FqP>();
  for (uint32_t i = tid; i < nv; i += VFY_THREADS) {
    uint32_t kk[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) kk[j] = scalars[((size_t)b * nv + i) * 8 + j];
    Xyzz<FqP> t = xyzz_mul_scalar(xyzz_from_affine(aff_load(pts + (size_t)b * nv + i)), kk);
    acc = xyzz_add(acc, t);
  }
  sh[tid] = acc;
  __syncthreads();
  for (uint32_t d = VFY_THREADS >> 1; d > 0; d >>= 1) {
    if (tid < d) sh[tid] = xyzz_add(sh[tid], sh[tid + d]);
    __syncthreads();
  }
  if (tid == 0) {
    Xyzz<FqP> tot = sh[0];
    xyzz_add_mixed(tot, aff_load(fixed_part + b));
    ok[b] = xyzz_is_identity(tot) ? 1 : 0;
  }
}

struct Verifier {
  Ctx* C; VkImpl& vk; uint32_t B;
  const bzh::Field& F; const bzh::Field& Fq;
  cudaStream_t st;
  Verifier(Ctx* c, VkImpl& v, uint32_t b) : C(c), vk(v), B(b), F(c->fp), Fq(c->fq), st(c->stream) {}

  // host evaluation of one postfix expression at the claimed openings
  HFe eval_expr(uint32_t lo, uint32_t hi, const std::vector<HFe>& ev, const std::map<std::pair<int, int>, int>& aq,
                const std::map<std::pair<int, int>, int>& fq, const std::map<std::pair<int, int>, int>& iq, int e_adv0, int e_fix0) const {
    const CircuitCopy& cs = vk.cs;
    std::vector<HFe> stck;
    for (uint32_t t = lo; t < hi; ++t) {
      const Token& k = cs.tokens[t];
      switch (k.op) {
        case 0: stck.push_back(cs.consts[k.a]); break;
        case 1: stck.push_back(ev[e_adv0 + aq.at({(int)k.a, k.b})]); break;
        case 2: stck.push_back(ev[e_fix0 + fq.at({(int)k.a, k.b})]); break;
        case 3: stck.push_back(ev[iq.at({(int)k.a, k.b})]); break;
        case 4: stck.back() = F.neg(stck.back()); break;
        case 5: { HFe r = stck.back(); stck.pop_back(); stck.back() = F.add(stck.back(), r); break; }
        case 6: { HFe r = stck.back(); stck.pop_back(); stck.back() = F.mul(stck.back(), r); break; }
        case 7: stck.back() = F.mul(stck.back(), cs.consts[k.a]); break;
        default: throw Error(-1, "bad token op");
      }
    }
    return stck.back();
  }

  void run(const void* instances, const uint32_t* instance_lens, uint32_t instance_stride, const uint8_t* proofs, uint32_t proof_len, uint8_t* results);
};

void Verifier::run(const void* instances, const uint32_t* instance_lens, uint32_t instance_stride, const uint8_t* proofs, uint32_t proof_len, uint8_t* results) {
  const CircuitCopy& cs = vk.cs;
  const uint32_t G = cs.G, I = cs.I, L = vk.L, bf = cs.bf, n = vk.n, k = cs.k, nsets = vk.nsets, qdeg = vk.qdeg;
  const uint32_t nps = (uint32_t)vk.point_sets.size();
  for (uint32_t b = 0; b < B; ++b) results[b] = 0;
  if (proof_len != vk.proof_size) return;                                  // short read / trailing bytes: Err
  for (uint32_t i = 0; i < I; ++i) if (instance_lens[i] > vk.usable) return;   // Error::InstanceTooLarge
  ParamsImpl& pr = *vk.params;
  if (vk.vk_fixed_comm.size() + vk.vk_perm_comm.size() != (size_t)(cs.F + vk.M) * 8) throw Error(BZ_ERR_INVALID, "internal: vk commitments missing");
  // ---- layout of the proof: which 32-byte items are points
  const uint32_t nev = vk.nev;
  std::vector<uint32_t> pt_off;        // byte offsets of the compressed points, in reading order
  uint32_t off = 0;
  auto take_pts = [&](uint32_t c) { for (uint32_t i = 0; i < c; ++i) { pt_off.push_back(off); off += 32; } };
  take_pts(G); take_pts(2 * L); take_pts(nsets); take_pts(L); take_pts(1); take_pts(qdeg);
  const uint32_t off_evals = off; off += 32 * nev;
  take_pts(1);                                     // q'
  const uint32_t off_uevals = off; off += 32 * nps;
  take_pts(1);                                     // S
  take_pts(2 * k);                                 // L_j, R_j
  const uint32_t off_c = off; off += 64;
  BZ_CHECK(off == vk.proof_size, "internal: proof layout mismatch");
  const uint32_t NP = (uint32_t)pt_off.size();
  // ---- device: decompress every point of every proof; instance commitments
  std::vector<uint8_t> comp((size_t)B * NP * 32);
  for (uint32_t b = 0; b < B; ++b)
    for (uint32_t i = 0; i < NP; ++i) memcpy(&comp[((size_t)b * NP + i) * 32], proofs + (size_t)b * proof_len + pt_off[i], 32);
  DevBuf &d_comp = vk.vwork[0], &d_pts = vk.vwork[1], &d_stat = vk.vwork[2], &d_inst = vk.vwork[3], &d_ptrs = vk.vwork[4], &d_extra = vk.vwork[5], &d_icomm = vk.vwork[6];
  d_comp.ensure(comp.size()); d_pts.ensure((size_t)B * NP * 64); d_stat.ensure((size_t)B * NP);
  BZ_CUDA(cudaMemcpyAsync(d_comp.p, comp.data(), comp.size(), cudaMemcpyHostToDevice, st));
  decompress_points_run(C, pr.curve, d_comp.p, d_pts.p, (uint8_t*)d_stat.p, B * NP);
  std::vector<uint64_t> h_pts((size_t)B * NP * 8), h_icomm((size_t)B * std::max(1u, I) * 8);
  std::vector<uint8_t> h_stat((size_t)B * NP);
  BZ_CUDA(cudaMemcpyAsync(h_pts.data(), d_pts.p, h_pts.size() * 8, cudaMemcpyDeviceToHost, st));
  BZ_CUDA(cudaMemcpyAsync(h_stat.data(), d_stat.p, h_stat.size(), cudaMemcpyDeviceToHost, st));
  if (I) {
    d_inst.ensure((size_t)B * I * n * 32); d_extra.ensure((size_t)B * I * 64); d_icomm.ensure((size_t)B * I * 64);
    BZ_CUDA(cudaMemsetAsync(d_inst.p, 0, (size_t)B * I * n * 32, st));
    std::vector<void*> mainp((size_t)B * I), extrap((size_t)B * I);
    std::vector<HFe> ex((size_t)B * I * 2, F.zero());
    for (uint32_t b = 0; b < B; ++b)
      for (uint32_t i = 0; i < I; ++i) {
        const size_t j = (size_t)b * I + i;
        if (instance_lens[i])
          BZ_CUDA(cudaMemcpyAsync((char*)d_inst.p + j * n * 32, (const char*)instances + j * instance_stride * 32, (size_t)instance_lens[i] * 32, cudaMemcpyDefault, st));
        mainp[j] = (char*)d_inst.p + j * n * 32; extrap[j] = (char*)d_extra.p + j * 64; ex[2 * j] = F.one();
      }
    BZ_CUDA(cudaMemcpyAsync(d_extra.p, ex.data(), ex.size() * 32, cudaMemcpyHostToDevice, st));
    const void* const* d = upload_msm_ptrs(C, d_ptrs, mainp, extrap);
    params_commit_run(C, pr, true, d, d + B * I, B * I, d_icomm.p);
    BZ_CUDA(cudaMemcpyAsync(h_icomm.data(), d_icomm.p, (size_t)B * I * 64, cudaMemcpyDeviceToHost, st));
  }
  BZ_CUDA(cudaStreamSynchronize(st));

  // ---- host: transcript and scalars, proof by proof
  std::map<std::pair<int, int>, int> aqm, fqm, iqm;
  for (size_t i = 0; i < cs.aq.size(); ++i) aqm[{cs.aq[i].first, cs.aq[i].second}] = (int)i;
  for (size_t i = 0; i < cs.fq.size(); ++i) fqm[{cs.fq[i].first, cs.fq[i].second}] = (int)i;
  for (size_t i = 0; i < cs.iq.size(); ++i) iqm[{cs.iq[i].first, cs.iq[i].second}] = (int)i;
  const int e_adv0 = (int)cs.iq.size(), e_fix0 = e_adv0 + (int)cs.aq.size(), e_rand = e_fix0 + (int)cs.fq.size(), e_sig0 = e_rand + 1;
  const int e_perm0 = e_sig0 + (int)vk.M, e_lk0 = e_perm0 + (nsets ? 3 * (int)nsets - 1 : 0);
  // variable points of the final check, per proof: every cmap commitment (h expands into its qdeg pieces), q', S, L_j, R_j
  uint32_t NV = 0;
  for (auto& ci : vk.cmap) NV += ci.cid == cid_h ? qdeg : 1;
  NV += 2 + 2 * k;
  std::vector<uint64_t> v_pts((size_t)B * NV * 8, 0), v_scal((size_t)B * NV * 4, 0);
  const uint32_t cstride = 2 + k;
  std::vector<HFe> s_consts((size_t)B * cstride, F.zero()), fx_extra((size_t)B * 2, F.zero());
  std::vector<uint8_t> alive(B, 1);
  const HFe one = F.one(), n_inv = F.inv(F.from_u64(n));
  for (uint32_t b = 0; b < B; ++b) {
    const uint8_t* proof = proofs + (size_t)b * proof_len;
    bool okp = true;
    for (uint32_t i = 0; i < NP; ++i) if (h_stat[(size_t)b * NP + i]) okp = false;     // from_bytes failed, or the identity (cannot be absorbed)
    if (!okp) { alive[b] = 0; continue; }
    ProofState ps;
    uint8_t sink[64]; ps.out = sink;
    uint32_t next_pt = 0;
    auto point_mont = [&](uint32_t idx) { return &h_pts[((size_t)b * NP + idx) * 8]; };
    auto read_point = [&]() { HostPoint hp; affine_to_host(Fq, point_mont(next_pt), hp); t_common_point(ps, hp); return next_pt++; };
    auto read_scalar = [&](uint32_t byte_off, HFe& out) {
      uint64_t raw[4]; memcpy(raw, proof + byte_off, 32);
      if (F.geq_mod(raw)) return false;                   // from_repr rejects non-canonical encodings
      out = F.from_raw(raw);
      t_common_scalar(ps, F, out);
      return true;
    };
    t_common_scalar(ps, F, cs.vk_repr);
    for (uint32_t i = 0; i < I; ++i) {
      HostPoint hp; affine_to_host(Fq, &h_icomm[((size_t)b * I + i) * 8], hp);
      if (hp.identity) { okp = false; break; }
      t_common_point(ps, hp);
    }
    if (!okp) { alive[b] = 0; continue; }
    std::vector<uint32_t> adv_pt(G), lkA(L), lkS(L), pz_pt(nsets), lkz_pt(L), h_pt(qdeg);
    for (uint32_t g = 0; g < G; ++g) adv_pt[g] = read_point();
    const HFe theta = t_squeeze(ps, F);
    for (uint32_t l = 0; l < L; ++l) { lkA[l] = read_point(); lkS[l] = read_point(); }
    const HFe beta = t_squeeze(ps, F), gamma = t_squeeze(ps, F);
    for (uint32_t s2 = 0; s2 < nsets; ++s2) pz_pt[s2] = read_point();
    for (uint32_t l = 0; l < L; ++l) lkz_pt[l] = read_point();
    const uint32_t rand_pt = read_point();
    const HFe y = t_squeeze(ps, F);
    for (uint32_t i = 0; i < qdeg; ++i) h_pt[i] = read_point();
    const HFe x = t_squeeze(ps, F);
    std::vector<HFe> ev(nev);
    for (uint32_t i = 0; i < nev && okp; ++i) okp = read_scalar(off_evals + 32 * i, ev[i]);
    if (!okp) { alive[b] = 0; continue; }
    // ---- expected h(x)
    HFe xn = x; for (uint32_t i = 0; i < k; ++i) xn = F.sqr(xn);
    const HFe xn_m1 = F.sub(xn, one);
    std::vector<HFe> w_is, inv1;                     // rotations -(bf+1) .. 0; one inversion for (x - w_i)..., (x^n - 1)
    for (int rot = -((int)bf + 1); rot <= 0; ++rot) { w_is.push_back(F.pow_u64(vk.omega_inv, (uint64_t)(-rot))); inv1.push_back(F.sub(x, w_is.back())); }
    inv1.push_back(xn_m1);
    host_batch_invert(F, inv1);
    std::vector<HFe> l_evals;
    for (size_t i = 0; i < w_is.size(); ++i) l_evals.push_back(F.mul(F.mul(F.mul(w_is[i], xn_m1), n_inv), inv1[i]));
    const HFe xn_m1_inv = inv1.back();
    const HFe l_last = l_evals[0], l_0 = l_evals[bf + 1];
    HFe l_blind = F.zero();
    for (uint32_t i = 1; i <= bf; ++i) l_blind = F.add(l_blind, l_evals[i]);
    const HFe one_minus = F.sub(one, F.add(l_last, l_blind));
    auto leaf_col = [&](std::pair<uint32_t, uint32_t> col) {
      if (col.first == 0) return ev[e_adv0 + aqm.at({(int)col.second, 0})];
      if (col.first == 1) return ev[e_fix0 + fqm.at({(int)col.second, 0})];
      return ev[iqm.at({(int)col.second, 0})];
    };
    HFe expected_h = F.zero();
    auto fold = [&](const HFe& e) { expected_h = F.add(F.mul(expected_h, y), e); };
    for (size_t g = 0; g + 1 < cs.gate_off.size(); ++g) fold(eval_expr(cs.gate_off[g], cs.gate_off[g + 1], ev, aqm, fqm, iqm, e_adv0, e_fix0));
    if (nsets) {
      auto pe = [&](uint32_t s2, int which) { return ev[e_perm0 + 3 * s2 + which]; };
      fold(F.mul(l_0, F.sub(one, pe(0, 0))));
      const HFe zl = pe(nsets - 1, 0);
      fold(F.mul(l_last, F.sub(F.sqr(zl), zl)));
      for (uint32_t s2 = 1; s2 < nsets; ++s2) fold(F.mul(F.sub(pe(s2, 0), pe(s2 - 1, 2)), l_0));
      const HFe delta = F.delta();
      for (uint32_t s2 = 0; s2 < nsets; ++s2) {
        const uint32_t c0 = s2 * vk.chunk_len, c1 = std::min<uint32_t>(vk.M, c0 + vk.chunk_len);
        HFe left = pe(s2, 1), right = pe(s2, 0);
        HFe cur_delta = F.mul(F.mul(beta, x), F.pow_u64(delta, c0));
        for (uint32_t j = c0; j < c1; ++j) {
          const HFe v = leaf_col(cs.perm[j]);
          left = F.mul(left, F.add(F.add(v, F.mul(beta, ev[e_sig0 + j])), gamma));
          right = F.mul(right, F.add(F.add(v, cur_delta), gamma));
          cur_delta = F.mul(cur_delta, delta);
        }
        fold(F.mul(F.sub(left, right), one_minus));
      }
    }
    for (uint32_t l = 0; l < L; ++l) {
      const int e = e_lk0 + 5 * (int)l;
      const HFe z = ev[e], z_next = ev[e + 1], a = ev[e + 2], a_inv = ev[e + 3], s = ev[e + 4];
      auto compress = [&](const std::vector<std::pair<uint32_t, uint32_t>>& es) {
        HFe acc = F.zero();
        for (auto& r : es) acc = F.add(F.mul(acc, theta), eval_expr(r.first, r.second, ev, aqm, fqm, iqm, e_adv0, e_fix0));
        return acc;
      };
      fold(F.mul(l_0, F.sub(one, z)));
      fold(F.mul(l_last, F.sub(F.sqr(z), z)));
      const HFe left = F.mul(F.mul(z_next, F.add(a, beta)), F.add(s, gamma));
      const HFe right = F.mul(F.mul(z, F.add(compress(cs.lookups[l].inputs), beta)), F.add(compress(cs.lookups[l].tables), gamma));
      fold(F.mul(F.sub(left, right), one_minus));
      fold(F.mul(l_0, F.sub(a, s)));
      fold(F.mul(F.mul(F.sub(a, s), F.sub(a, a_inv)), one_minus));
    }
    expected_h = F.mul(expected_h, xn_m1_inv);
    // ---- multiopen verifier
    const HFe x1 = t_squeeze(ps, F), x2 = t_squeeze(ps, F);
    auto rot_point = [&](int r) { return r >= 0 ? F.mul(x, F.pow_u64(vk.omega, (uint64_t)r)) : F.mul(x, F.pow_u64(vk.omega_inv, (uint64_t)(-r))); };
    // evaluation of every commitment at every point of its set
    std::vector<std::vector<std::vector<HFe>>> c_evals(vk.cmap.size());
    for (size_t ci = 0; ci < vk.cmap.size(); ++ci) c_evals[ci].assign(1, std::vector<HFe>(vk.point_sets[vk.cmap[ci].set].size(), F.zero()));
    for (const Query& q : vk.queries) {
      size_t ci = 0;
      while (vk.cmap[ci].cid != q.cid) ++ci;
      const std::vector<int>& set = vk.point_sets[vk.cmap[ci].set];
      const size_t j = std::find(set.begin(), set.end(), q.rot) - set.begin();
      c_evals[ci][0][j] = q.eval_idx >= 0 ? ev[q.eval_idx] : expected_h;
    }
    std::vector<std::vector<HFe>> q_eval_sets(nps);
    for (uint32_t s2 = 0; s2 < nps; ++s2) q_eval_sets[s2].assign(vk.point_sets[s2].size(), F.zero());
    std::vector<HFe> comm_scalar(vk.cmap.size(), one);         // x1 power inside its set
    {
      std::vector<HFe> set_pow(nps, one);
      for (int ci = (int)vk.cmap.size() - 1; ci >= 0; --ci) { comm_scalar[ci] = set_pow[vk.cmap[ci].set]; set_pow[vk.cmap[ci].set] = F.mul(set_pow[vk.cmap[ci].set], x1); }
    }
    for (size_t ci = 0; ci < vk.cmap.size(); ++ci) {
      std::vector<HFe>& qs = q_eval_sets[vk.cmap[ci].set];
      for (size_t j = 0; j < qs.size(); ++j) qs[j] = F.add(F.mul(qs[j], x1), c_evals[ci][0][j]);
    }
    const uint32_t qprime_pt = read_point();
    const HFe x3 = t_squeeze(ps, F);
    std::vector<HFe> u_evals(nps);
    for (uint32_t s2 = 0; s2 < nps && okp; ++s2) okp = read_scalar(off_uevals + 32 * s2, u_evals[s2]);
    if (!okp) { alive[b] = 0; continue; }
    HFe msm_eval = F.zero();
    {
      // lagrange_interpolate(points, evals)(x3) per set: all denominators of all sets share one inversion
      std::vector<std::vector<HFe>> pts(nps), nums(nps);
      std::vector<HFe> inv2;
      for (uint32_t s2 = 0; s2 < nps; ++s2) {
        for (int r : vk.point_sets[s2]) pts[s2].push_back(rot_point(r));
        HFe den = one;
        for (size_t j = 0; j < pts[s2].size(); ++j) {
          HFe num = one, dj = one;
          for (size_t m2 = 0; m2 < pts[s2].size(); ++m2) if (m2 != j) { num = F.mul(num, F.sub(x3, pts[s2][m2])); dj = F.mul(dj, F.sub(pts[s2][j], pts[s2][m2])); }
          nums[s2].push_back(num); inv2.push_back(dj);
          den = F.mul(den, F.sub(x3, pts[s2][j]));
        }
        inv2.push_back(den);
      }
      host_batch_invert(F, inv2);
      size_t at = 0;
      for (uint32_t s2 = 0; s2 < nps; ++s2) {
        HFe r_eval = F.zero();
        for (size_t j = 0; j < pts[s2].size(); ++j) r_eval = F.add(r_eval, F.mul(F.mul(q_eval_sets[s2][j], nums[s2][j]), inv2[at++]));
        msm_eval = F.add(F.mul(msm_eval, x2), F.mul(F.sub(u_evals[s2], r_eval), inv2[at++]));
      }
    }
    const HFe x4 = t_squeeze(ps, F);
    HFe v = msm_eval;
    for (uint32_t s2 = 0; s2 < nps; ++s2) v = F.add(F.mul(v, x4), u_evals[s2]);
    std::vector<HFe> x4pow(nps + 1, one);
    for (uint32_t i = 1; i <= nps; ++i) x4pow[i] = F.mul(x4pow[i - 1], x4);
    // ---- IPA verifier
    const uint32_t s_pt = read_point();
    const HFe xi = t_squeeze(ps, F), z = t_squeeze(ps, F);
    std::vector<uint32_t> l_pt(k), r_pt(k);
    std::vector<HFe> us(k);
    for (uint32_t j = 0; j < k; ++j) { l_pt[j] = read_point(); r_pt[j] = read_point(); us[j] = t_squeeze(ps, F); }
    HFe c_sc, f_sc;
    okp = read_scalar(off_c, c_sc) && read_scalar(off_c + 32, f_sc);
    if (!okp) { alive[b] = 0; continue; }
    HFe bb = one, cur = x3;
    for (int j = (int)k - 1; j >= 0; --j) { bb = F.mul(bb, F.add(one, F.mul(us[j], cur))); cur = F.sqr(cur); }
    // ---- scalars of the final check
    uint64_t* vp = &v_pts[(size_t)b * NV * 8];
    uint64_t* vs = &v_scal[(size_t)b * NV * 4];
    uint32_t nvi = 0;
    auto push = [&](const uint64_t* mont_pt, const HFe& sc) { memcpy(vp + (size_t)nvi * 8, mont_pt, 64); F.to_raw(sc, vs + (size_t)nvi * 4); ++nvi; };
    for (size_t ci = 0; ci < vk.cmap.size(); ++ci) {
      const int cid = vk.cmap[ci].cid;
      const HFe sc = F.mul(comm_scalar[ci], x4pow[nps - 1 - vk.cmap[ci].set]);
      if (cid == cid_h) { HFe p2 = sc; for (uint32_t i = 0; i < qdeg; ++i) { push(point_mont(h_pt[i]), p2); p2 = F.mul(p2, xn); } }
      else if (cid == cid_rand) push(point_mont(rand_pt), sc);
      else if (cid >= cid_sig) push(&vk.vk_perm_comm[(size_t)(cid - cid_sig) * 8], sc);
      else if (cid >= cid_fix) push(&vk.vk_fixed_comm[(size_t)(cid - cid_fix) * 8], sc);
      else if (cid >= cid_lk) { const uint32_t l = (cid - cid_lk) / 3, w = (cid - cid_lk) % 3; push(point_mont(w == 0 ? lkA[l] : w == 1 ? lkS[l] : lkz_pt[l]), sc); }
      else if (cid >= cid_pz) push(point_mont(pz_pt[cid - cid_pz]), sc);
      else if (cid >= cid_adv) push(point_mont(adv_pt[cid - cid_adv]), sc);
      else push(&h_icomm[((size_t)b * I + (cid - cid_inst)) * 8], sc);
    }
    push(point_mont(qprime_pt), x4pow[nps]);
    push(point_mont(s_pt), xi);
    std::vector<HFe> us_inv = us;
    host_batch_invert(F, us_inv);
    for (uint32_t j = 0; j < k; ++j) { push(point_mont(l_pt[j]), us_inv[j]); push(point_mont(r_pt[j]), us[j]); }
    BZ_CHECK(nvi == NV, "internal: verifier point count mismatch");
    HFe* sc = &s_consts[(size_t)b * cstride];
    sc[0] = F.neg(c_sc); sc[1] = F.neg(v);
    for (uint32_t i = 0; i < k; ++i) sc[2 + i] = us[k - 1 - i];
    fx_extra[2 * b] = F.neg(f_sc);                                   // W
    fx_extra[2 * b + 1] = F.neg(F.mul(F.mul(c_sc, bb), z));          // U
  }
  // ---- device: compute_s, the fixed-base part, the final check
  DevBuf &d_sc = vk.vwork[7], &d_s = vk.vwork[8], &d_fx = vk.vwork[9], &d_fptrs = vk.vwork[10], &d_fpart = vk.vwork[11], &d_vp = vk.vwork[12], &d_vs = vk.vwork[13], &d_ok = vk.vwork[14];
  d_sc.ensure(s_consts.size() * 32); d_s.ensure((size_t)B * n * 32); d_fx.ensure((size_t)B * 64);
  d_fpart.ensure((size_t)B * 64); d_vp.ensure(v_pts.size() * 8); d_vs.ensure(v_scal.size() * 8); d_ok.ensure(B);
  BZ_CUDA(cudaMemcpyAsync(d_sc.p, s_consts.data(), s_consts.size() * 32, cudaMemcpyHostToDevice, st));
  BZ_CUDA(cudaMemcpyAsync(d_fx.p, fx_extra.data(), fx_extra.size() * 32, cudaMemcpyHostToDevice, st));
  BZ_CUDA(cudaMemcpyAsync(d_vp.p, v_pts.data(), v_pts.size() * 8, cudaMemcpyHostToDevice, st));
  BZ_CUDA(cudaMemcpyAsync(d_vs.p, v_scal.data(), v_scal.size() * 8, cudaMemcpyHostToDevice, st));
  compute_s_kernel<<<dim3((n + 127) / 128, B), 128, 0, st>>>((const DFe*)d_sc.p, cstride, (DFe*)d_s.p, k);
  C->kernel_launches++;
  std::vector<void*> mainp(B), extrap(B);
  for (uint32_t b = 0; b < B; ++b) { mainp[b] = (char*)d_s.p + (size_t)b * n * 32; extrap[b] = (char*)d_fx.p + (size_t)b * 64; }
  const void* const* d = upload_msm_ptrs(C, d_fptrs, mainp, extrap);
  params_commit_run(C, pr, false, d, d + B, B, d_fpart.p);
  verify_final_kernel<<<B, VFY_THREADS, 0, st>>>((const Affine<FqP>*)d_vp.p, (const uint32_t*)d_vs.p, NV, (const Affine<FqP>*)d_fpart.p, (uint8_t*)d_ok.p);
  C->kernel_launches++;
  std::vector<uint8_t> h_ok(B);
  BZ_CUDA(cudaMemcpyAsync(h_ok.data(), d_ok.p, B, cudaMemcpyDeviceToHost, st));
  BZ_CUDA(cudaStreamSynchronize(st));
  BZ_CUDA(cudaGetLastError());
  for (uint32_t b = 0; b < B; ++b) results[b] = (alive[b] && h_ok[b]) ? 1 : 0;
}

}  // namespace bz

namespace bz {

static void check_verify_args(const VkImpl& vk, const void* instances, const uint32_t* instance_lens, uint32_t instance_stride) {
  BZ_CHECK(vk.cs.I == 0 || (instances && instance_lens), "instances missing");
  for (uint32_t i = 0; i < vk.cs.I; ++i) BZ_CHECK(instance_lens[i] <= instance_stride, "instance_lens[i] exceeds instance_stride");
}

// keygen_vk's commitments as the caller hands them over: `count` affine points (x || y, Montgomery).  A real vk never holds the
// identity (keygen_vk commits with Blind::default(), which adds [1]W), and the final check takes its bases as affine points.
static void take_commitments(const bzh::Field& Fq, const void* src, uint32_t count, const char* what, std::vector<uint64_t>& dst) {
  dst.resize((size_t)count * 8);
  if (count) memcpy(dst.data(), src, dst.size() * 8);
  const HFe five = Fq.from_u64(5);
  for (uint32_t i = 0; i < count; ++i) {
    const uint64_t* p = &dst[(size_t)i * 8];
    const std::string at = std::string(what) + " commitment " + std::to_string(i);
    BZ_CHECK(!Fq.geq_mod(p) && !Fq.geq_mod(p + 4), at + ": coordinate not canonical (>= q)");
    HFe x, y; memcpy(x.l, p, 32); memcpy(y.l, p + 4, 32);
    BZ_CHECK(!(x.is_zero() && y.is_zero()), at + " is the identity");
    BZ_CHECK(Fq.sqr(y) == Fq.add(Fq.mul(Fq.sqr(x), x), five), at + " is not on y^2 = x^3 + 5");
  }
}

}  // namespace bz

extern "C" API int bz_verify_proofs(bz_ctx* ctx, bz_pk* pkh, uint32_t batch, const void* instances, const uint32_t* instance_lens,
                                    uint32_t instance_stride, const void* proofs, uint32_t proof_len, uint8_t* results) {
  PV_TRY(ctx, {
    BZ_CHECK(pkh && proofs && results && batch >= 1, "null argument");
    PkImpl& pk = pkh->p;
    check_verify_args(pk, instances, instance_lens, instance_stride);
    if (pk.vk_fixed_comm.size() + pk.vk_perm_comm.size() != (size_t)(pk.cs.F + pk.M) * 8) {
      int rc = bz_pk_vk_commitments(ctx, pkh, nullptr, nullptr);
      if (rc != BZ_OK) return rc;
    }
    Verifier vf(C, pk, batch);
    vf.run(instances, instance_lens, instance_stride, (const uint8_t*)proofs, proof_len, results);
  });
}

extern "C" API int bz_vk_create(bz_ctx* ctx, bz_params* params, const bz_circuit* cin, const void* fixed_commitments,
                                const void* perm_commitments, bz_vk** out) {
  PV_TRY(ctx, {
    BZ_CHECK(out && params && cin, "null argument");
    *out = nullptr;
    BZ_CHECK(params->p.curve == 0, "verifying key: only the Vesta commitment curve (circuits over pallas::Base) is wired up");
    BZ_CHECK(cin->k == params->p.k, "circuit k != params k");
    BZ_CHECK(fixed_commitments || !cin->num_fixed, "null fixed_commitments");
    BZ_CHECK(perm_commitments || !cin->n_perm_columns, "null perm_commitments");
    std::unique_ptr<bz_vk> h(new bz_vk());
    VkImpl& vk = h->v;
    vk.params = &params->p;
    vk_host_setup(C->fp, vk, cin);
    take_commitments(C->fq, fixed_commitments, vk.cs.F, "fixed", vk.vk_fixed_comm);
    take_commitments(C->fq, perm_commitments, vk.M, "permutation", vk.vk_perm_comm);
    *out = h.release();
  });
}

extern "C" API void bz_vk_destroy(bz_vk* vk) { delete vk; }
extern "C" API uint32_t bz_vk_proof_size(const bz_vk* vk) { return vk ? vk->v.proof_size : 0; }

extern "C" API int bz_verify_proofs_vk(bz_ctx* ctx, bz_vk* vkh, uint32_t batch, const void* instances, const uint32_t* instance_lens,
                                       uint32_t instance_stride, const void* proofs, uint32_t proof_len, uint8_t* results) {
  PV_TRY(ctx, {
    BZ_CHECK(vkh && proofs && results && batch >= 1, "null argument");
    VkImpl& vk = vkh->v;
    check_verify_args(vk, instances, instance_lens, instance_stride);
    Verifier vf(C, vk, batch);
    vf.run(instances, instance_lens, instance_stride, (const uint8_t*)proofs, proof_len, results);
  });
}
