// Radix-2^k number-theoretic transforms over Fp / Fq for sm_100a.
// Replaces halo2_proofs 0.2.0 `arithmetic::best_fft` and the `EvaluationDomain` wrappers
// `lagrange_to_coeff`, `coeff_to_extended`, `extended_to_coeff` (U: src/arithmetic.rs,
// src/poly/domain.rs; SURVEY §8 a4/a5).  Natural order in, natural order out (same contract as
// best_fft), so results are bit-identical field elements.
//
// Decomposition: N = N1*N2(*N3).  Every pass runs 2^logL-point transforms on "lines" of the array
// that are staged in shared memory (two 16-byte planes per element -> conflict-free LDS.128),
// multiplies by the inter-pass twiddles w_M^(k*t) and writes the line back through an arbitrary
// (u, v, k) stride map, which is how the four-step transposes are folded into the passes: no
// separate bit-reversal or transpose pass ever touches HBM.  N <= 2^12 is a single pass (one read,
// one write = the algorithmic 64*N bytes); up to 2^20..2^24 are two/three passes.
// Fusions: zero-padding + zeta^(i mod 3) coset pre-scale on the first pass (coeff_to_extended),
// N^-1 and zeta^-(i mod 3) post-scale on the last pass (ifft / extended_to_coeff).
#include "common.h"
#include "field.cuh"

namespace bz {

template <class P> struct NttPassArgs {
  const Fe<P>* in;
  Fe<P>* out;
  uint32_t logL, logT, logV;
  uint64_t in_u, in_v, in_k;
  uint64_t out_u, out_v, out_k;
  uint64_t in_batch, out_batch;
  uint64_t in_batch2, out_batch2;     // second (outer) batch dimension: blockIdx.z
  const Fe<P>* wsmall;
  uint32_t tw_logM;
  const Fe<P>* tw_lo;
  const Fe<P>* tw_hi;
  uint32_t k_limit;
  uint32_t zero_stages;              // zero-padded lines: the first log2(L / k_limit) stages only replicate (their second operand is 0)
  uint32_t pre_mode;
  uint32_t post_mode;
  Fe<P> pre[3];
  Fe<P> post[3];
};

template <class P> __device__ __forceinline__ Fe<P> sm_ld(const uint4* p0, const uint4* p1, uint32_t i) {
  uint4 a = p0[i], b = p1[i];
  Fe<P> r;
  r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
  r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
  return r;
}
template <class P> __device__ __forceinline__ void sm_st(uint4* p0, uint4* p1, uint32_t i, const Fe<P>& v) {
  p0[i] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
  p1[i] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

constexpr uint32_t TW_FULL_LOG = 16;     // inter-pass twiddles w_M^e: one table of M entries up to 2^16 (2 MB, L2 resident), lo/hi split above

template <class P>
__global__ void __launch_bounds__(512) ntt_pass_kernel(const __grid_constant__ NttPassArgs<P> a) {
  extern __shared__ uint4 smem[];
  const uint32_t logL = a.logL, logT = a.logT;
  const uint32_t L = 1u << logL, T = 1u << logT, tile = L << logT;
  uint4* p0 = smem;
  uint4* p1 = smem + tile;
  const uint32_t tid = threadIdx.x, nth = blockDim.x;
  const uint64_t line0 = (uint64_t)blockIdx.x << logT;
  const uint64_t u = line0 >> a.logV, v0 = line0 & ((1ull << a.logV) - 1);
  const uint64_t in_off0 = u * a.in_u + v0 * a.in_v;
  const Fe<P>* in = a.in + (uint64_t)blockIdx.z * a.in_batch2 + (uint64_t)blockIdx.y * a.in_batch + in_off0;

  // ---- load (bit-reversed placement), fused zero-pad / coset pre-scale ----
  for (uint32_t idx = tid; idx < tile; idx += nth) {
    uint32_t k, line;
    if (a.in_k == 1) { k = idx & (L - 1); line = idx >> logL; }
    else { line = idx & (T - 1); k = idx >> logT; }
    Fe<P> x = fe_zero<P>();
    if (k < a.k_limit) {
      uint64_t off = (uint64_t)line * a.in_v + (uint64_t)k * a.in_k;
      x = fe_load(in + off);
      if (a.pre_mode) {
        uint32_t m3 = (uint32_t)((in_off0 + off) % 3);
        if (m3) x = fe_mul(x, a.pre[m3]);
      }
    }
    uint32_t slot = logL ? (__brev(k) >> (32 - logL)) : 0;
    sm_st<P>(p0, p1, (slot << logT) + line, x);
  }
  __syncthreads();

  // ---- log2(L) butterfly stages in shared memory ----
  for (uint32_t s = 0; s < logL; ++s) {
    const uint32_t d = 1u << s;
    for (uint32_t idx = tid; idx < (tile >> 1); idx += nth) {
      uint32_t line = idx & (T - 1), b = idx >> logT;
      uint32_t pos = b & (d - 1), grp = b >> s;
      uint32_t i0 = ((grp << (s + 1)) + pos) << logT | line;
      uint32_t i1 = i0 + (d << logT);
      Fe<P> x = sm_ld<P>(p0, p1, i0);
      if (s < a.zero_stages) { sm_st<P>(p0, p1, i1, x); continue; }          // x + 0*w, x - 0*w
      Fe<P> y = sm_ld<P>(p0, p1, i1);
      if (pos) y = fe_mul(y, fe_load(a.wsmall + ((uint64_t)pos << (WSMALL_LOG - 1 - s))));
      sm_st<P>(p0, p1, i0, fe_add(x, y));
      sm_st<P>(p0, p1, i1, fe_sub(x, y));
    }
    __syncthreads();
  }

  // ---- store through the output stride map, fused inter-pass twiddle / post-scale ----
  const uint64_t out_off0 = u * a.out_u + v0 * a.out_v;
  Fe<P>* out = a.out + (uint64_t)blockIdx.z * a.out_batch2 + (uint64_t)blockIdx.y * a.out_batch + out_off0;
  for (uint32_t idx = tid; idx < tile; idx += nth) {
    uint32_t k, line;
    if (a.out_k == 1) { k = idx & (L - 1); line = idx >> logL; }
    else { line = idx & (T - 1); k = idx >> logT; }
    Fe<P> x = sm_ld<P>(p0, p1, (k << logT) + line);
    if (a.tw_logM) {
      uint64_t e = (uint64_t)k * (v0 + line);       // < M by construction
      if (e) {
        if (a.tw_logM <= TW_FULL_LOG) x = fe_mul(x, fe_load(a.tw_lo + e));
        else {
          uint32_t elo = (uint32_t)(e & 4095), ehi = (uint32_t)(e >> 12);
          if (elo) x = fe_mul(x, fe_load(a.tw_lo + elo));
          if (ehi) x = fe_mul(x, fe_load(a.tw_hi + ehi));
        }
      }
    }
    uint64_t off = (uint64_t)line * a.out_v + (uint64_t)k * a.out_k;
    if (a.post_mode == 1) x = fe_mul(x, a.post[0]);
    else if (a.post_mode == 3) x = fe_mul(x, a.post[(out_off0 + off) % 3]);
    fe_store(out + off, x);
  }
}

// out[i] = base^(i * mult), i < n
template <class P> __global__ void pow_table_kernel(Fe<P>* out, Fe<P> base, uint32_t n, uint64_t mult) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  fe_store(out + i, fe_pow_u64<P>(base, (uint64_t)i * mult));
}

template <class P> static Fe<P> to_dev(const bzh::Fe& h) {
  Fe<P> r;
  memcpy(r.l, h.l, 32);
  return r;
}

static bzh::Fe omega_for(const bzh::Field& F, int logM, bool inverse) {
  bzh::Fe w = F.root_of_unity();
  for (int i = logM; i < 32; ++i) w = F.sqr(w);
  return inverse ? F.inv(w) : w;
}

template <class P> static const Fe<P>* get_wsmall(Ctx* ctx, int field, bool inverse) {
  DevBuf& b = ctx->wsmall[field][inverse ? 1 : 0];
  if (!b.p) {
    const uint32_t n = 1u << (WSMALL_LOG - 1);
    b.alloc((size_t)n * 32);
    bzh::Fe w = omega_for(ctx->field(field), WSMALL_LOG, inverse);
    pow_table_kernel<P><<<(n + 127) / 128, 128, 0, ctx->stream>>>(b.as<Fe<P>>(), to_dev<P>(w), n, 1);
    ctx->kernel_launches++;
    BZ_CUDA(cudaGetLastError());
  }
  return b.as<Fe<P>>();
}

template <class P> static const NttTable& get_tw(Ctx* ctx, int field, bool inverse, int logM) {
  NttTableKey key{field, inverse ? 1 : 0, logM};
  auto it = ctx->ntt_tables.find(key);
  if (it != ctx->ntt_tables.end()) return it->second;
  NttTable& t = ctx->ntt_tables[key];
  bzh::Fe w = omega_for(ctx->field(field), logM, inverse);
  uint32_t nlo = logM <= (int)TW_FULL_LOG ? (1u << logM) : 4096u;
  t.lo.alloc((size_t)nlo * 32);
  pow_table_kernel<P><<<(nlo + 127) / 128, 128, 0, ctx->stream>>>(t.lo.as<Fe<P>>(), to_dev<P>(w), nlo, 1);
  ctx->kernel_launches++;
  if (logM > (int)TW_FULL_LOG) {
    uint32_t nhi = 1u << (logM - 12);
    t.hi.alloc((size_t)nhi * 32);
    pow_table_kernel<P><<<(nhi + 127) / 128, 128, 0, ctx->stream>>>(t.hi.as<Fe<P>>(), to_dev<P>(w), nhi, 4096);
    ctx->kernel_launches++;
  }
  BZ_CUDA(cudaGetLastError());
  return t;
}

template <class P> static void launch_pass(Ctx* ctx, NttPassArgs<P>& a, uint64_t nlines, int batch, int batch2) {
  uint32_t tile = 1u << (a.logL + a.logT);
  a.zero_stages = 0;
  if (a.k_limit && a.k_limit < (1u << a.logL) && (a.k_limit & (a.k_limit - 1)) == 0)
    while ((a.k_limit << a.zero_stages) < (1u << a.logL)) ++a.zero_stages;
  size_t smem = (size_t)tile * 32;
  int threads = tile >= 4096 ? 512 : (tile >= 512 ? 256 : (tile >= 64 ? (int)tile / 2 : 32));
  static PerDeviceOnce once;            // per template instantiation
  once.run(ctx->device, [] { cudaFuncSetAttribute(ntt_pass_kernel<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024); });
  dim3 grid((unsigned)(nlines >> a.logT), (unsigned)batch, (unsigned)batch2);
  ProfScope prof(ctx, PROF_NTT_PASS);
  ntt_pass_kernel<P><<<grid, threads, smem, ctx->stream>>>(a);
  ctx->kernel_launches++;
  BZ_CUDA(cudaGetLastError());
}

template <class P>
static void ntt_run_t(Ctx* ctx, int field, const Fe<P>* in, Fe<P>* out, int logN, bool inverse, int batch, const NttFusion& fu,
                      int batch2, uint64_t in_stride2, uint64_t out_stride2) {
  BZ_CHECK(logN >= 0 && logN <= 30, "ntt: logN out of range");
  const bzh::Field& F = ctx->field(field);
  const uint64_t N = 1ull << logN;
  const uint64_t n_in = fu.n_in ? fu.n_in : N;
  BZ_CHECK((n_in & (n_in - 1)) == 0 && n_in <= N, "ntt: n_in must be a power of two <= N");

  NttPassArgs<P> base{};
  base.wsmall = get_wsmall<P>(ctx, field, inverse);
  // fusion constants
  Fe<P> pre[3], post[3];
  bzh::Fe zeta = F.zeta(), zeta2 = F.sqr(zeta);
  pre[0] = to_dev<P>(F.one()); pre[1] = to_dev<P>(zeta); pre[2] = to_dev<P>(zeta2);
  if (fu.post_mode) {
    bzh::Fe ninv = F.inv(F.from_u64(N));
    post[0] = to_dev<P>(ninv);
    post[1] = to_dev<P>(F.mul(ninv, zeta2));   // zeta^-1 = zeta^2
    post[2] = to_dev<P>(F.mul(ninv, zeta));    // zeta^-2 = zeta
  }
  for (int i = 0; i < 3; ++i) { base.pre[i] = pre[i]; base.post[i] = post[i]; }

  int npass = logN <= 12 ? 1 : (logN <= 20 ? 2 : 3);      // two passes above 2^20 were probed and dropped (DESIGN.md section 6)
  if (npass == 1) {
    NttPassArgs<P> a = base;
    a.in = in; a.out = out;
    a.logL = logN; a.logT = 0; a.logV = 0;
    a.in_u = a.in_v = 0; a.in_k = 1; a.out_u = a.out_v = 0; a.out_k = 1;
    a.in_batch = n_in; a.out_batch = N;
    a.tw_logM = 0;
    a.k_limit = (uint32_t)n_in;
    a.pre_mode = fu.pre_zeta ? 1 : 0;
    a.post_mode = fu.post_mode;
    a.in_batch2 = in_stride2; a.out_batch2 = out_stride2;
    launch_pass<P>(ctx, a, 1, batch, batch2);
    return;
  }
  ctx->ntt_tmp.ensure((size_t)batch * batch2 * N * 32);
  const uint64_t tmp_stride2 = (uint64_t)batch * N;
  Fe<P>* tmp = ctx->ntt_tmp.as<Fe<P>>();
  if (npass == 2) {
    int l1 = (logN + 1) / 2, l2 = logN - l1;
    uint64_t N1 = 1ull << l1, N2 = 1ull << l2;
    BZ_CHECK(n_in >= N2 || n_in == N, "ntt: zero-padded input too short for this decomposition");
    const NttTable& tw = get_tw<P>(ctx, field, inverse, logN);
    {  // pass A: N2 strided lines of length N1, twiddle w_N^(k*j2)
      NttPassArgs<P> a = base;
      a.in = in; a.out = tmp;
      a.logL = l1; a.logV = l2; a.logT = (uint32_t)std::min<int>(l2, std::max(0, 11 - l1));
      a.in_u = 0; a.in_v = 1; a.in_k = N2; a.out_u = 0; a.out_v = 1; a.out_k = N2;
      a.in_batch = n_in; a.out_batch = N;
      a.tw_logM = logN; a.tw_lo = tw.lo.as<Fe<P>>(); a.tw_hi = tw.hi.as<Fe<P>>();
      a.k_limit = (uint32_t)(n_in == N ? N1 : n_in / N2);
      a.pre_mode = fu.pre_zeta ? 1 : 0; a.post_mode = 0;
      a.in_batch2 = in_stride2; a.out_batch2 = tmp_stride2;
      launch_pass<P>(ctx, a, N2, batch, batch2);
    }
    {  // pass B: N1 contiguous lines of length N2, output index k1 + N1*k2
      NttPassArgs<P> a = base;
      a.in = tmp; a.out = out;
      a.logL = l2; a.logV = l1; a.logT = (uint32_t)std::min<int>(l1, std::max(0, 11 - l2));
      a.in_u = 0; a.in_v = N2; a.in_k = 1; a.out_u = 0; a.out_v = 1; a.out_k = N1;
      a.in_batch = N; a.out_batch = N;
      a.tw_logM = 0; a.k_limit = (uint32_t)N2; a.pre_mode = 0; a.post_mode = fu.post_mode;
      a.in_batch2 = tmp_stride2; a.out_batch2 = out_stride2;
      launch_pass<P>(ctx, a, N1, batch, batch2);
    }
    return;
  }
  // three passes: N = N1*N2*N3
  int l1 = (logN + 2) / 3, l2 = (logN - l1 + 1) / 2, l3 = logN - l1 - l2;
  uint64_t N1 = 1ull << l1, N2 = 1ull << l2, N3 = 1ull << l3, N23 = N2 * N3;
  BZ_CHECK(n_in >= N23 || n_in == N, "ntt: zero-padded input too short for this decomposition");
  const NttTable& twN = get_tw<P>(ctx, field, inverse, logN);
  const NttTable& tw23 = get_tw<P>(ctx, field, inverse, l2 + l3);
  {  // pass A
    NttPassArgs<P> a = base;
    a.in = in; a.out = tmp;
    a.logL = l1; a.logV = l2 + l3; a.logT = (uint32_t)std::max(0, 11 - l1);
    a.in_u = 0; a.in_v = 1; a.in_k = N23; a.out_u = 0; a.out_v = 1; a.out_k = N23;
    a.in_batch = n_in; a.out_batch = N;
    a.tw_logM = logN; a.tw_lo = twN.lo.as<Fe<P>>(); a.tw_hi = twN.hi.as<Fe<P>>();
    a.k_limit = (uint32_t)(n_in == N ? N1 : n_in / N23);
    a.pre_mode = fu.pre_zeta ? 1 : 0; a.post_mode = 0;
    a.in_batch2 = in_stride2; a.out_batch2 = tmp_stride2;
    launch_pass<P>(ctx, a, N23, batch, batch2);
  }
  {  // pass B1: lines (u = k1, v = j3), length N2 at stride N3, twiddle w_{N2N3}^(k*j3), in place
    NttPassArgs<P> a = base;
    a.in = tmp; a.out = tmp;
    a.logL = l2; a.logV = l3; a.logT = (uint32_t)std::min<int>(l3, std::max(0, 11 - l2));
    a.in_u = N23; a.in_v = 1; a.in_k = N3; a.out_u = N23; a.out_v = 1; a.out_k = N3;
    a.in_batch = N; a.out_batch = N;
    a.tw_logM = l2 + l3; a.tw_lo = tw23.lo.as<Fe<P>>(); a.tw_hi = tw23.hi.as<Fe<P>>();
    a.k_limit = (uint32_t)N2; a.pre_mode = 0; a.post_mode = 0;
    a.in_batch2 = tmp_stride2; a.out_batch2 = tmp_stride2;
    launch_pass<P>(ctx, a, N1 * N3, batch, batch2);
  }
  {  // pass B2: lines (u = k2, v = k1), contiguous length N3, output index k1 + N1*k2 + N1*N2*k3
    NttPassArgs<P> a = base;
    a.in = tmp; a.out = out;
    a.logL = l3; a.logV = l1; a.logT = (uint32_t)std::min<int>(l1, std::max(0, 11 - l3));
    a.in_u = N3; a.in_v = N23; a.in_k = 1; a.out_u = N1; a.out_v = 1; a.out_k = N1 * N2;
    a.in_batch = N; a.out_batch = N;
    a.tw_logM = 0; a.k_limit = (uint32_t)N3; a.pre_mode = 0; a.post_mode = fu.post_mode;
    a.in_batch2 = tmp_stride2; a.out_batch2 = out_stride2;
    launch_pass<P>(ctx, a, N1 * N2, batch, batch2);
  }
}

void ntt_run(Ctx* ctx, int field, const void* in, void* out, int logN, bool inverse, int batch, const NttFusion& fu,
             int batch2, uint64_t in_stride2, uint64_t out_stride2) {
  if (batch <= 0 || batch2 <= 0) return;
  if (field == 0) ntt_run_t<FpP>(ctx, field, (const Fe<FpP>*)in, (Fe<FpP>*)out, logN, inverse, batch, fu, batch2, in_stride2, out_stride2);
  else ntt_run_t<FqP>(ctx, field, (const Fe<FqP>*)in, (Fe<FqP>*)out, logN, inverse, batch, fu, batch2, in_stride2, out_stride2);
}

}  // namespace bz
