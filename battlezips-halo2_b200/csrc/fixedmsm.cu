// Fixed-base multi-scalar multiplication for `Params::commit` / `Params::commit_lagrange` and the IPA
// L/R terms (U: halo2_proofs 0.2.0 src/poly/commitment.rs, src/poly/commitment/prover.rs; SURVEY §8 a3/a11).
//
// B200-first design: every commitment of every proof uses one of two fixed bases (g || w || u  or
// g_lagrange || w), so with 180 GB of HBM we tabulate ALL signed-digit multiples
//     T[w][d-1][i] = d * 2^(c*w) * B_i ,  d = 1 .. 2^(c-1),  w < ceil(256/c)
// once per Params (affine, 64 B per entry; a few GB).  A commitment is then a flat sum of at most
// ceil(256/c) * (n+1) table entries: no buckets, no sorting, no doublings, no bucket reduction, and
// zero digits (witness columns are mostly 0/1) cost nothing.  One launch commits a whole batch of
// polynomials.  All arithmetic is IMAD-pipe Montgomery work in XYZZ coordinates.
#include "common.h"
#include "curve.cuh"
#include "fixedmsm.h"
#include <cstdlib>

namespace bz {

// ---- table construction (one-off per Params) -----------------------------------------------------
// scratch[d][i] = (d + 1) * base[i] for d < nbk.  The multiples of one point form a chain of mixed additions; the chain is
// cut into `nseg` segments that start from [seg * len] base[i] (a 32-bit double-and-add), so a 2^11-point URS still fills
// the GPU: thread = (segment, point), adjacent threads store adjacent points.
template <class BP>
__global__ void fb_multiples_kernel(const Affine<BP>* __restrict__ base, uint32_t npts, uint32_t nbk, uint32_t nseg, Xyzz<BP>* __restrict__ scratch) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (uint64_t)npts * nseg) return;
  const uint32_t i = (uint32_t)(t % npts), seg = (uint32_t)(t / npts), len = nbk / nseg, d0 = seg * len;
  Affine<BP> p = aff_load(base + i);
  Xyzz<BP> acc = d0 ? xyzz_mul_u32(xyzz_from_affine(p), d0) : xyzz_identity<BP>();
  for (uint32_t d = d0; d < d0 + len; ++d) {
    xyzz_add_mixed(acc, p);
    Xyzz<BP>* o = scratch + (size_t)d * npts + i;
    fe_store(&o->x, acc.x); fe_store(&o->y, acc.y); fe_store(&o->zz, acc.zz); fe_store(&o->zzz, acc.zzz);
  }
}

// XYZZ -> affine with Montgomery's trick over RUN consecutive entries per thread
template <class BP, int RUN>
__global__ void fb_to_affine_kernel(const Xyzz<BP>* __restrict__ in, Affine<BP>* __restrict__ out, uint64_t total) {
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t lo = t * RUN;
  if (lo >= total) return;
  uint32_t cnt = (uint32_t)min((uint64_t)RUN, total - lo);
  Fe<BP> pre[RUN];
  Fe<BP> acc = fe_one<BP>();
  for (uint32_t j = 0; j < cnt; ++j) {
    pre[j] = acc;
    Fe<BP> z = fe_load(&in[lo + j].zzz);
    if (!fe_is_zero(z)) acc = fe_mul(acc, z);
  }
  Fe<BP> inv = fe_inv(acc);
  for (int j = (int)cnt - 1; j >= 0; --j) {
    const Xyzz<BP>* q = in + lo + j;
    Fe<BP> zzz = fe_load(&q->zzz);
    Affine<BP> r;
    if (fe_is_zero(zzz)) { r.x = fe_zero<BP>(); r.y = fe_zero<BP>(); }
    else {
      Fe<BP> zi3 = fe_mul(inv, pre[j]);        // 1/zzz
      inv = fe_mul(inv, zzz);
      Fe<BP> zz = fe_load(&q->zz);
      Fe<BP> zi2 = fe_mul(fe_mul(fe_sqr(zi3), zz), zz);   // zzz^-2 * zz^2 = 1/zz
      r.x = fe_mul(fe_load(&q->x), zi2);
      r.y = fe_mul(fe_load(&q->y), zi3);
    }
    fe_store(&out[lo + j].x, r.x); fe_store(&out[lo + j].y, r.y);
  }
}

// next window's base: 2 * (2^(c-1) * P) -> affine
template <class BP>
__global__ void fb_next_base_kernel(const Xyzz<BP>* __restrict__ scratch_last, Affine<BP>* __restrict__ base, uint32_t npts) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npts) return;
  const Xyzz<BP>* q = scratch_last + i;
  Xyzz<BP> v; v.x = fe_load(&q->x); v.y = fe_load(&q->y); v.zz = fe_load(&q->zz); v.zzz = fe_load(&q->zzz);
  Affine<BP> r = xyzz_to_affine(xyzz_dbl(v));
  fe_store(&base[i].x, r.x); fe_store(&base[i].y, r.y);
}

template <class BP>
static void fb_build_t(Ctx* ctx, FixedBase& fb, const void* bases_dev) {
  cudaStream_t st = ctx->stream;
  const uint32_t npts = fb.npts, nbk = fb.nbk, W = fb.W;
  fb.table.alloc((size_t)W * nbk * npts * sizeof(Affine<BP>));
  DevBuf scratch, base;
  scratch.alloc((size_t)nbk * npts * sizeof(Xyzz<BP>));
  base.alloc((size_t)npts * sizeof(Affine<BP>));
  BZ_CUDA(cudaMemcpyAsync(base.p, bases_dev, (size_t)npts * sizeof(Affine<BP>), cudaMemcpyDeviceToDevice, st));
  const uint64_t per_window = (uint64_t)nbk * npts;
  uint32_t nseg = 1;                                   // power of two (divides nbk): ~128 K threads, segments of >= 64 additions
  while (nseg * 2 <= nbk / 64 && (uint64_t)npts * nseg * 2 <= 131072) nseg *= 2;
  for (uint32_t w = 0; w < W; ++w) {
    fb_multiples_kernel<BP><<<(unsigned)(((uint64_t)npts * nseg + 63) / 64), 64, 0, st>>>(base.as<Affine<BP>>(), npts, nbk, nseg, scratch.as<Xyzz<BP>>());
    uint64_t nthreads = (per_window + 15) / 16;
    fb_to_affine_kernel<BP, 16><<<(unsigned)((nthreads + 127) / 128), 128, 0, st>>>(
        scratch.as<Xyzz<BP>>(), fb.table.as<Affine<BP>>() + (size_t)w * per_window, per_window);
    if (w + 1 < W)
      fb_next_base_kernel<BP><<<(npts + 63) / 64, 64, 0, st>>>(scratch.as<Xyzz<BP>>() + (size_t)(nbk - 1) * npts, base.as<Affine<BP>>(), npts);
    ctx->kernel_launches += 3;
  }
  BZ_CUDA(cudaGetLastError());
  BZ_CUDA(cudaStreamSynchronize(st));
}

void fixed_base_build(Ctx* ctx, FixedBase& fb, int curve, const void* bases_dev, uint32_t npts, uint32_t c) {
  BZ_CHECK(c >= 4 && c <= 16, "fixed-base window out of range");
  BZ_CHECK((uint64_t)((256 + c - 1) / c) * (1ull << (c - 1)) * npts < (1ull << 31), "fixed-base table too large for 31-bit entry indices");
  fb.curve = curve; fb.npts = npts; fb.c = c; fb.W = (256 + c - 1) / c; fb.nbk = 1u << (c - 1);
  if (curve == 0) fb_build_t<FqP>(ctx, fb, bases_dev); else fb_build_t<FpP>(ctx, fb, bases_dev);
}

// ---- the commitment pipeline ------------------------------------------------------------------------
// MSM m sums over points [0, npts): scalars of points i < n_main come from main[m] (a polynomial, Montgomery form),
// the trailing npts - n_main points (w, u: blinds / IPA cross terms) from extra[m] (may be null = zero).
//
//   1. fb_decode_kernel   one thread per (msm, point): signed digits -> packed table indices, appended to the MSM's
//                         entry list (warp-aggregated atomic reservation; zero digits vanish here, so witness columns
//                         -- mostly 0/1 -- cost only what they contain)
//   2. fb_accumulate_kernel   ONE resident wave of threads; the entries of all MSMs of the launch form a flat index
//                         space cut into equal shares, one per thread: gather + mixed additions, no barriers in the
//                         loop, every warp full, every SM busy until the end
//   3. fb_fold_kernel     one CTA per MSM: strided sum of its partials, shared-memory tree, affine output
constexpr int FB_THREADS = 128;
constexpr int FB_FOLD_THREADS = 128;          // batched calls (many MSMs per launch)
constexpr int FB_FOLD_THREADS_WIDE = 512;     // few MSMs per launch (single-proof latency): more threads per fold

template <class SP>
__global__ void __launch_bounds__(FB_THREADS) fb_decode_kernel(uint32_t npts, uint32_t c, uint32_t W, uint32_t nbk,
                                 const Fe<SP>* const* __restrict__ main, uint32_t n_main, const Fe<SP>* const* __restrict__ extra,
                                 uint32_t* __restrict__ lists, uint32_t list_stride, uint32_t* __restrict__ list_count) {
  const uint32_t m = blockIdx.y, i = blockIdx.x * FB_THREADS + threadIdx.x, lane = threadIdx.x & 31;
  const uint32_t half = 1u << (c - 1), full = 1u << c;
  Fe<SP> s = fe_zero<SP>();
  bool have = false;
  if (i < npts) {
    const Fe<SP>* se = extra ? extra[m] : nullptr;
    if (i < n_main) { s = fe_load(main[m] + i); have = true; }
    else if (se) { s = fe_load(se + (i - n_main)); have = true; }
  }
  uint32_t cnt = 0;
  if (have && !fe_is_zero(s)) {
    s = fe_from_mont(s);
    uint32_t carry = 0;
    for (uint32_t w = 0; w < W; ++w) {
      uint32_t bit = w * c, limb = bit >> 5, sh_ = bit & 31;
      uint32_t raw = 0;
      if (limb < 8) {
        raw = s.l[limb] >> sh_;
        if (sh_ + c > 32 && limb + 1 < 8) raw |= s.l[limb + 1] << (32 - sh_);
        raw &= full - 1;
      }
      uint32_t v = raw + carry;
      carry = v > half ? 1u : 0u;
      cnt += (v != 0 && v != full) ? 1u : 0u;
    }
  } else have = false;
  // warp-aggregated reservation in this MSM's list
  uint32_t incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { uint32_t o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= (uint32_t)d) incl += o; }
  uint32_t warp_total = __shfl_sync(0xffffffffu, incl, 31), base = 0;
  if (lane == 31 && warp_total) base = atomicAdd(&list_count[m], warp_total);
  base = __shfl_sync(0xffffffffu, base, 31);
  if (!have) return;
  uint32_t* list = lists + (size_t)m * list_stride;
  uint32_t off = base + incl - cnt, carry = 0;
  for (uint32_t w = 0; w < W; ++w) {
    uint32_t bit = w * c, limb = bit >> 5, sh_ = bit & 31;
    uint32_t raw = 0;
    if (limb < 8) {
      raw = s.l[limb] >> sh_;
      if (sh_ + c > 32 && limb + 1 < 8) raw |= s.l[limb + 1] << (32 - sh_);
      raw &= full - 1;
    }
    uint32_t v = raw + carry;
    bool neg = v > half;
    uint32_t d = neg ? full - v : v;
    carry = neg ? 1u : 0u;
    if (d) list[off++] = (uint32_t)(((size_t)w * nbk + (d - 1)) * npts + i) | (neg ? 0x80000000u : 0u);
  }
}

// Exclusive prefix sum of the per-MSM entry counts into shared memory (every CTA recomputes it: n_msm <= FB_MAX_MSM words),
// and the balanced share q = entries per thread.  All entries of all MSMs of a launch form ONE flat index space that is
// cut into equal ranges, one per resident thread: no wave quantisation (r1d ncu: the per-segment grid ran 2.16 waves on
// the IPA-round launches and left the fma pipe at 56-66 %), and ~8x fewer partial sums to fold.
constexpr uint32_t FB_MAX_MSM = 4096;
constexpr uint32_t FB_MIN_SHARE = 16;
__device__ __forceinline__ uint32_t fb_plan(const uint32_t* __restrict__ list_count, uint32_t n_msm, uint32_t total_threads, uint32_t* off /* [n_msm + 1] shared */,
                                            uint32_t* wsum /* [33] shared */) {
  const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
  const uint32_t per = (n_msm + blockDim.x - 1) / blockDim.x, lo = min(tid * per, n_msm), hi = min(lo + per, n_msm);
  uint32_t s = 0;
  for (uint32_t i = lo; i < hi; ++i) s += list_count[i];
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
  for (uint32_t i = lo; i < hi; ++i) { off[i] = run; run += list_count[i]; }
  const uint32_t total = wsum[32];
  if (tid == 0) off[n_msm] = total;
  __syncthreads();
  return max(FB_MIN_SHARE, (total + total_threads - 1) / total_threads);
}

// Warp W owns the flat entries [W*32q, (W+1)*32q); inside every MSM piece of that range lane l takes entries l, l+32, ...
// (coalesced list reads) and keeps its own sum.  The table point of the NEXT entry is gathered before the current
// addition starts, so the list -> table dependent DRAM round trips overlap the ~10 field multiplications of the addition.
// A warp emits 32 partials per MSM it touches, at index (W + m)*32 + lane (unique and increasing along the flat order).
template <class BP>
__global__ void __launch_bounds__(FB_THREADS, 4) fb_accumulate_kernel(const Affine<BP>* __restrict__ table, const uint32_t* __restrict__ lists,
                                 uint32_t list_stride, const uint32_t* __restrict__ list_count, uint32_t n_msm,
                                 Xyzz<BP>* __restrict__ partial, unsigned long long* __restrict__ add_counter) {
  extern __shared__ uint32_t fb_off[];
  __shared__ uint32_t wsum[33];
  const uint32_t T = gridDim.x * FB_THREADS, t = blockIdx.x * FB_THREADS + threadIdx.x, lane = threadIdx.x & 31, W = t >> 5;
  const uint32_t q = fb_plan(list_count, n_msm, T, fb_off, wsum);
  const uint32_t total = fb_off[n_msm];
  const uint64_t base64 = (uint64_t)W * 32u * q;
  uint32_t my_adds = 0;
  if (base64 < total) {
    const uint32_t base = (uint32_t)base64, end = (uint32_t)min((uint64_t)total, base64 + (uint64_t)32 * q);
    uint32_t lo = 0, hi = n_msm;                     // m = last MSM with off[m] <= base
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (fb_off[mid] <= base) lo = mid; else hi = mid; }
    uint32_t m = lo, pbeg = base;
    while (pbeg < end) {
      while (fb_off[m + 1] <= pbeg) ++m;               // skip MSMs without entries
      const uint32_t pend = min(end, fb_off[m + 1]);
      const uint32_t* list = lists + (size_t)m * list_stride - fb_off[m];
      Xyzz<BP> acc = xyzz_identity<BP>();
      uint32_t p = pbeg + lane;
      uint32_t ent = 0, ent_n = 0;
      Affine<BP> pt;
      if (p < pend) { ent = list[p]; pt = aff_load(table + (ent & 0x7fffffffu)); }
      if (p + 32 < pend) ent_n = list[p + 32];
      while (p < pend) {
        const bool more = p + 32 < pend;
        Affine<BP> pt_n;
        uint32_t ent_nn = 0;
        if (more) pt_n = aff_load(table + (ent_n & 0x7fffffffu));
        if (p + 64 < pend) ent_nn = list[p + 64];
        xyzz_add_mixed_signed(acc, pt, (ent >> 31) != 0);
        ++my_adds;
        if (more) pt = pt_n;
        ent = ent_n; ent_n = ent_nn;
        p += 32;
      }
      Xyzz<BP>* o = partial + ((size_t)W + m) * 32 + lane;
      fe_store(&o->x, acc.x); fe_store(&o->y, acc.y); fe_store(&o->zz, acc.zz); fe_store(&o->zzz, acc.zzz);
      pbeg = pend;
    }
  }
  if (add_counter) {       // profiling only: exact number of mixed additions this launch performed
    uint32_t tot = __reduce_add_sync(0xffffffffu, my_adds);
    if ((threadIdx.x & 31) == 0 && tot) atomicAdd(add_counter, (unsigned long long)tot);
  }
}

// fold the partials of each MSM and normalise: one CTA per MSM -> affine (64 B), identity = zeros
template <class BP, bool XYZZ_OUT, int THREADS>
__global__ void __launch_bounds__(THREADS) fb_fold_kernel(const Xyzz<BP>* __restrict__ partial, const uint32_t* __restrict__ list_count,
                                 uint32_t n_msm, uint32_t acc_threads, void* __restrict__ out_v) {
  __shared__ uint32_t wsum[33];
  extern __shared__ uint32_t fb_off[];
  Xyzz<BP>* sh = reinterpret_cast<Xyzz<BP>*>(fb_off + (((size_t)n_msm + 1 + 31) & ~size_t(31)));      // after the offsets, 128 B aligned
  const uint32_t m = blockIdx.x, tid = threadIdx.x;
  const uint32_t q = fb_plan(list_count, n_msm, acc_threads, fb_off, wsum);
  const uint32_t lo = fb_off[m], hi = fb_off[m + 1];
  Xyzz<BP> acc = xyzz_identity<BP>();
  if (hi > lo) {
    const uint32_t w_first = lo / (32u * q), w_last = (hi - 1) / (32u * q);
    const uint32_t npieces = (w_last - w_first + 1) * 32u;         // warp w, lane l -> (w + m) * 32 + l : contiguous
    for (uint32_t t = tid; t < npieces; t += THREADS) {
      const Xyzz<BP>* p = partial + ((size_t)w_first + m) * 32 + t;
      Xyzz<BP> v; v.x = fe_load(&p->x); v.y = fe_load(&p->y); v.zz = fe_load(&p->zz); v.zzz = fe_load(&p->zzz);
      acc = xyzz_add(acc, v);
    }
  }
  sh[tid] = acc;
  __syncthreads();
  for (uint32_t d = THREADS >> 1; d > 0; d >>= 1) {
    if (tid < d) sh[tid] = xyzz_add(sh[tid], sh[tid + d]);
    __syncthreads();
  }
  if (tid == 0) {
    if (XYZZ_OUT) {
      Xyzz<BP>* o = reinterpret_cast<Xyzz<BP>*>(out_v) + m;
      fe_store(&o->x, sh[0].x); fe_store(&o->y, sh[0].y); fe_store(&o->zz, sh[0].zz); fe_store(&o->zzz, sh[0].zzz);
    } else {
      Affine<BP>* out = reinterpret_cast<Affine<BP>*>(out_v);
      Affine<BP> r = xyzz_to_affine(sh[0]);
      fe_store(&out[m].x, r.x); fe_store(&out[m].y, r.y);
    }
  }
}

// Few MSMs per launch (one large proof: 1 - 2 MSMs of 2^16+ points): a single CTA per MSM would fold all ~75 000 thread partials
// of the accumulate wave alone (150 serial additions per thread, 0.8 ms per call at k = 18 -- as long as the accumulation
// itself).  Two levels instead: G CTAs per MSM fold a slice each, then one small CTA per MSM folds the G slice sums.
constexpr int FB_PREFOLD_THREADS = 256;
template <class BP>
__global__ void __launch_bounds__(FB_PREFOLD_THREADS) fb_prefold_kernel(const Xyzz<BP>* __restrict__ partial, const uint32_t* __restrict__ list_count,
                                 uint32_t n_msm, uint32_t acc_threads, Xyzz<BP>* __restrict__ slice_sums) {
  __shared__ uint32_t wsum[33];
  extern __shared__ uint32_t fb_off[];
  Xyzz<BP>* sh = reinterpret_cast<Xyzz<BP>*>(fb_off + (((size_t)n_msm + 1 + 31) & ~size_t(31)));
  const uint32_t m = blockIdx.x, g = blockIdx.y, G = gridDim.y, tid = threadIdx.x;
  const uint32_t q = fb_plan(list_count, n_msm, acc_threads, fb_off, wsum);
  const uint32_t lo = fb_off[m], hi = fb_off[m + 1];
  Xyzz<BP> acc = xyzz_identity<BP>();
  if (hi > lo) {
    const uint32_t w_first = lo / (32u * q), w_last = (hi - 1) / (32u * q);
    const uint32_t npieces = (w_last - w_first + 1) * 32u, per = (npieces + G - 1) / G;
    const uint32_t t_end = min(npieces, (g + 1) * per);
    for (uint32_t t = g * per + tid; t < t_end; t += FB_PREFOLD_THREADS) {
      const Xyzz<BP>* p = partial + ((size_t)w_first + m) * 32 + t;
      Xyzz<BP> v; v.x = fe_load(&p->x); v.y = fe_load(&p->y); v.zz = fe_load(&p->zz); v.zzz = fe_load(&p->zzz);
      acc = xyzz_add(acc, v);
    }
  }
  sh[tid] = acc;
  __syncthreads();
  for (uint32_t d = FB_PREFOLD_THREADS >> 1; d > 0; d >>= 1) {
    if (tid < d) sh[tid] = xyzz_add(sh[tid], sh[tid + d]);
    __syncthreads();
  }
  if (tid == 0) {
    Xyzz<BP>* o = slice_sums + (size_t)m * G + g;
    fe_store(&o->x, sh[0].x); fe_store(&o->y, sh[0].y); fe_store(&o->zz, sh[0].zz); fe_store(&o->zzz, sh[0].zzz);
  }
}
// G (a power of two <= 64) threads per MSM
template <class BP, bool XYZZ_OUT>
__global__ void __launch_bounds__(64) fb_fold_slices_kernel(const Xyzz<BP>* __restrict__ slice_sums, void* __restrict__ out_v) {
  __shared__ Xyzz<BP> sh[64];
  const uint32_t m = blockIdx.x, tid = threadIdx.x, G = blockDim.x;
  const Xyzz<BP>* p = slice_sums + (size_t)m * G + tid;
  Xyzz<BP> v; v.x = fe_load(&p->x); v.y = fe_load(&p->y); v.zz = fe_load(&p->zz); v.zzz = fe_load(&p->zzz);
  sh[tid] = v;
  __syncthreads();
  for (uint32_t d = G >> 1; d > 0; d >>= 1) {
    if (tid < d) sh[tid] = xyzz_add(sh[tid], sh[tid + d]);
    __syncthreads();
  }
  if (tid == 0) {
    if (XYZZ_OUT) {
      Xyzz<BP>* o = reinterpret_cast<Xyzz<BP>*>(out_v) + m;
      fe_store(&o->x, sh[0].x); fe_store(&o->y, sh[0].y); fe_store(&o->zz, sh[0].zz); fe_store(&o->zzz, sh[0].zzz);
    } else {
      Affine<BP>* out = reinterpret_cast<Affine<BP>*>(out_v);
      Affine<BP> r = xyzz_to_affine(sh[0]);
      fe_store(&out[m].x, r.x); fe_store(&out[m].y, r.y);
    }
  }
}

template <class BP, class SP>
static void fixed_msm_run_t(Ctx* ctx, const FixedBase& fb, const void* const* d_main, uint32_t n_main, const void* const* d_extra,
                            uint32_t n_msm, void* d_out, bool xyzz_out) {
  cudaStream_t st = ctx->stream;
  if (!ctx->counters.p) { ctx->counters.alloc(64); BZ_CUDA(cudaMemsetAsync(ctx->counters.p, 0, 64, st)); }
  const uint32_t list_stride = fb.npts * fb.W;                          // worst case: every digit non-zero
  static int ctas_dev[BZ_MAX_DEVICES];   // per template instantiation and device; several prover lanes (host threads) may race to set them
  static PerDeviceOnce once;
  const int dev = ctx->device >= 0 && ctx->device < BZ_MAX_DEVICES ? ctx->device : 0;
  once.run(ctx->device, [dev] {
    int ctas_per_sm = 0;
    cudaFuncSetAttribute(fb_accumulate_kernel<BP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((FB_MAX_MSM + 1) * 4));
    int v = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, fb_accumulate_kernel<BP>, FB_THREADS, (FB_MAX_MSM + 1) * 4);
    ctas_per_sm = v < 1 ? 1 : v;
    const int fold_smem = (int)((FB_MAX_MSM + 32) * 4 + FB_FOLD_THREADS_WIDE * sizeof(Xyzz<BP>));
    cudaFuncSetAttribute(fb_fold_kernel<BP, true, FB_FOLD_THREADS_WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, fold_smem);
    cudaFuncSetAttribute(fb_fold_kernel<BP, false, FB_FOLD_THREADS_WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, fold_smem);
    cudaFuncSetAttribute(fb_fold_kernel<BP, true, FB_FOLD_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, fold_smem);
    cudaFuncSetAttribute(fb_fold_kernel<BP, false, FB_FOLD_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, fold_smem);
    // BZ_FB_CTAS_PER_SM: fewer resident CTAs of the accumulate wave than fit (A/B: leaves registers for the other prover lanes' kernels)
    if (const char* e = getenv("BZ_FB_CTAS_PER_SM")) { const int v2 = atoi(e); if (v2 >= 1 && v2 < ctas_per_sm) ctas_per_sm = v2; }
    ctas_dev[dev] = ctas_per_sm;
  });
  const uint32_t acc_ctas = (uint32_t)ctx->sm_count * (uint32_t)ctas_dev[dev], acc_threads = acc_ctas * FB_THREADS;
  const uint32_t max_nm = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(FB_MAX_MSM, 0xffffffffull / list_stride));   // flat index fits 32 bits
  for (uint32_t m0 = 0; m0 < n_msm; m0 += max_nm) {
    const uint32_t nm = std::min(max_nm, n_msm - m0);
    ctx->scratch[0].ensure((size_t)nm * list_stride * 4);
    ctx->scratch[1].ensure((size_t)nm * 4 + 64);
    ctx->scratch[3].ensure(((size_t)acc_threads + 32 * (size_t)nm + 32 + 64 * 256) * sizeof(Xyzz<BP>));   // thread partials + slice sums of the two-level fold
    uint32_t* lists = ctx->scratch[0].as<uint32_t>();
    uint32_t* counts = ctx->scratch[1].as<uint32_t>();
    Xyzz<BP>* partial = ctx->scratch[3].as<Xyzz<BP>>();
    BZ_CUDA(cudaMemsetAsync(counts, 0, (size_t)nm * 4, st));
    unsigned long long* cnt = ctx->profiling ? (unsigned long long*)ctx->counters.p : nullptr;
    const size_t smem = ((size_t)nm + 1) * 4;
    {
      ProfScope p(ctx, PROF_FIXED_MSM);
      fb_decode_kernel<SP><<<dim3((fb.npts + FB_THREADS - 1) / FB_THREADS, nm), FB_THREADS, 0, st>>>(
          fb.npts, fb.c, fb.W, fb.nbk, (const Fe<SP>* const*)d_main + m0, n_main, d_extra ? (const Fe<SP>* const*)d_extra + m0 : nullptr, lists, list_stride, counts);
      fb_accumulate_kernel<BP><<<acc_ctas, FB_THREADS, smem, st>>>(fb.table.as<Affine<BP>>(), lists, list_stride, counts, nm, partial, cnt);
      // fold: offsets + one XYZZ slot per thread in dynamic shared memory.  A launch with many thread partials per MSM (a few large
      // MSMs: one big proof) folds in two levels, G CTAs per MSM first
      const uint64_t pieces_per_msm = ((uint64_t)acc_threads + 32 * (uint64_t)nm) / nm;
      uint32_t G = 1;
      while (G < 64 && nm * G < 256 && pieces_per_msm / (G * 2) >= 2 * FB_PREFOLD_THREADS) G *= 2;
      const bool wide = nm < 48;
      const size_t fsm = (((size_t)nm + 1 + 31) & ~size_t(31)) * 4 + (size_t)(wide ? FB_FOLD_THREADS_WIDE : FB_FOLD_THREADS) * sizeof(Xyzz<BP>);
      if (G > 1) {
        Xyzz<BP>* slice_sums = partial + (size_t)acc_threads + 32 * (size_t)nm + 32;
        const size_t psm = (((size_t)nm + 1 + 31) & ~size_t(31)) * 4 + (size_t)FB_PREFOLD_THREADS * sizeof(Xyzz<BP>);
        fb_prefold_kernel<BP><<<dim3(nm, G), FB_PREFOLD_THREADS, psm, st>>>(partial, counts, nm, acc_threads, slice_sums);
        if (xyzz_out) fb_fold_slices_kernel<BP, true><<<nm, G, 0, st>>>(slice_sums, (Xyzz<BP>*)d_out + m0);
        else fb_fold_slices_kernel<BP, false><<<nm, G, 0, st>>>(slice_sums, (Affine<BP>*)d_out + m0);
        ctx->kernel_launches += 1;
      } else if (wide) {
        if (xyzz_out) fb_fold_kernel<BP, true, FB_FOLD_THREADS_WIDE><<<nm, FB_FOLD_THREADS_WIDE, fsm, st>>>(partial, counts, nm, acc_threads, (Xyzz<BP>*)d_out + m0);
        else fb_fold_kernel<BP, false, FB_FOLD_THREADS_WIDE><<<nm, FB_FOLD_THREADS_WIDE, fsm, st>>>(partial, counts, nm, acc_threads, (Affine<BP>*)d_out + m0);
      } else {
        if (xyzz_out) fb_fold_kernel<BP, true, FB_FOLD_THREADS><<<nm, FB_FOLD_THREADS, fsm, st>>>(partial, counts, nm, acc_threads, (Xyzz<BP>*)d_out + m0);
        else fb_fold_kernel<BP, false, FB_FOLD_THREADS><<<nm, FB_FOLD_THREADS, fsm, st>>>(partial, counts, nm, acc_threads, (Affine<BP>*)d_out + m0);
      }
    }
    ctx->kernel_launches += 3;
  }
  BZ_CUDA(cudaGetLastError());
}

void fixed_msm_run(Ctx* ctx, const FixedBase& fb, const void* const* d_main, uint32_t n_main, const void* const* d_extra,
                   uint32_t n_msm, void* d_out, bool xyzz_out) {
  if (!n_msm) return;
  BZ_CHECK(n_main <= fb.npts, "fixed msm: more scalars than table points");
  if (fb.curve == 0) fixed_msm_run_t<FqP, FpP>(ctx, fb, d_main, n_main, d_extra, n_msm, d_out, xyzz_out);
  else fixed_msm_run_t<FpP, FqP>(ctx, fb, d_main, n_main, d_extra, n_msm, d_out, xyzz_out);
}

}  // namespace bz
