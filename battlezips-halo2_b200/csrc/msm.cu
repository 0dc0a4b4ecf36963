// Variable-base multi-scalar multiplication  sum_i s_i * B_i  over Vesta / Pallas for sm_100a.
// Replaces halo2_proofs 0.2.0 `arithmetic::best_multiexp` (U: src/arithmetic.rs; SURVEY §8 a2).
// The reference algorithm (per-thread chunks, unsigned ceil(ln n)-bit windows, serial buckets) is
// NOT followed: the result is a group element, canonical after to_affine, so any evaluation order
// is bit-exact (SURVEY §0 fact 5).  Here: signed-digit windows (2^(c-1) buckets per window),
// counting sort of (window, bucket) keys with L2 atomics (hand-written: histogram, scan, scatter -- no library sort), one accumulator per bucket in XYZZ
// coordinates (8M+2S mixed additions, complete formulas), chunk-parallel running-sum reduction
// per window and a final Horner over the windows.  Everything is integer-pipe work (IMAD); the
// only HBM traffic is 32 B/scalar + 64 B/point gathers.
#include "common.h"
#include "curve.cuh"

namespace bz {

// ---- 1. counting sort of the non-zero signed digits by (window, bucket).  The key of a digit is  window * nb + (|digit| - 1),
// its value the point index with the sign in bit 31.  Two passes over the scalars recompute the digits (one Montgomery
// multiplication per scalar) instead of materialising and radix-sorting W * n (key, value) pairs:
//   msm_hist_kernel     counts[key]++                      msm_scan_kernel (below)   offsets = exclusive scan of counts
//   msm_scatter_kernel  sorted[offsets[key] + slot] = value, slot handed out by an atomic cursor per bucket
// Lanes of a warp that hit the same bucket (witness-like scalars: a fifth of all scalars equal 1) are combined with
// __match_any_sync, so a hot bucket costs one atomic per warp instead of 32 serialised ones.  The order inside a bucket is
// whatever the atomics give; the bucket's SUM does not depend on it.
template <class SP, class F>
__device__ __forceinline__ void msm_for_each_digit(const Fe<SP>& canonical, uint32_t c, uint32_t W, uint32_t nb, F&& f) {
  uint32_t carry = 0;
  const uint32_t half = 1u << (c - 1), full = 1u << c;
  for (uint32_t w = 0; w < W; ++w) {
    const uint32_t bit = w * c, limb = bit >> 5, sh = bit & 31;
    uint32_t raw = 0;
    if (limb < 8) {
      raw = canonical.l[limb] >> sh;
      if (sh + c > 32 && limb + 1 < 8) raw |= canonical.l[limb + 1] << (32 - sh);
      raw &= full - 1;
    }
    const uint32_t v = raw + carry;
    const bool neg = v > half;
    const uint32_t d = neg ? full - v : v;
    carry = neg ? 1u : 0u;
    f(d ? w * nb + d - 1 : 0xffffffffu, neg);          // every lane calls f for every window (warp-synchronous inside)
  }
}

// Where the scalars of a batch of MSMs over the SAME bases live: one contiguous array (`single`), or per MSM a main polynomial of
// n_main scalars plus a few trailing extras (blinding factors; the U / W terms of the IPA) -- the layout the table MSM takes
// too.  `first` shifts the window for a point-range shard.
template <class SP> struct ScalarSrc {
  const Fe<SP>* single;
  const Fe<SP>* const* mains;
  const Fe<SP>* const* extras;
  uint32_t n_main, first;
  __device__ __forceinline__ Fe<SP> load(uint32_t m, uint32_t i) const {
    if (single) return fe_load(single + i);
    const uint32_t g = i + first;
    return g < n_main ? fe_load(mains[m] + g) : fe_load(extras[m] + (g - n_main));
  }
};

// grid = (ceil(n / 256), MSMs of the batch).  A batch is sorted as ONE problem with  MSMs x W  "virtual windows": the key of MSM m
// is shifted by m * W * nb, and everything downstream (scan, segments, bucket sums, window reduction) only sees more windows.
template <class SP>
__global__ void __launch_bounds__(256) msm_hist_kernel(ScalarSrc<SP> src, uint32_t n, uint32_t c, uint32_t W, uint32_t nb, uint32_t* __restrict__ counts) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31, m = blockIdx.y;
  counts += (size_t)m * W * nb;
  Fe<SP> s = fe_zero<SP>();
  if (i < n) s = fe_from_mont(src.load(m, i));
  msm_for_each_digit<SP>(s, c, W, nb, [&](uint32_t key, bool) {
    // uniform scalars: 32 distinct keys per warp, one atomic each.  Only when neighbouring lanes collide (skewed scalars) is the
    // warp's traffic to a bucket combined -- __match_any_sync costs one step per distinct key, too slow for the common case
    const uint32_t neighbour = __shfl_xor_sync(0xffffffffu, key, 1);      // unconditional: every lane takes part in the shuffle
    const bool dup = key != 0xffffffffu && key == neighbour;
    if (__any_sync(0xffffffffu, dup)) {
      const uint32_t peers = __match_any_sync(0xffffffffu, key);
      if (key != 0xffffffffu && lane == (uint32_t)(__ffs((int)peers) - 1)) atomicAdd(&counts[key], (uint32_t)__popc(peers));
    } else if (key != 0xffffffffu) atomicAdd(&counts[key], 1u);
  });
}

template <class SP>
__global__ void __launch_bounds__(256) msm_scatter_kernel(ScalarSrc<SP> src, uint32_t n, uint32_t c, uint32_t W, uint32_t nb,
                                                          uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31, m = blockIdx.y;
  cursor += (size_t)m * W * nb;
  Fe<SP> s = fe_zero<SP>();
  if (i < n) s = fe_from_mont(src.load(m, i));
  msm_for_each_digit<SP>(s, c, W, nb, [&](uint32_t key, bool neg) {
    const uint32_t neighbour = __shfl_xor_sync(0xffffffffu, key, 1);
    const bool dup = key != 0xffffffffu && key == neighbour;
    if (__any_sync(0xffffffffu, dup)) {
      const uint32_t peers = __match_any_sync(0xffffffffu, key);
      const uint32_t leader = (uint32_t)(__ffs((int)peers) - 1);
      uint32_t base = 0;
      if (key != 0xffffffffu && lane == leader) base = atomicAdd(&cursor[key], (uint32_t)__popc(peers));
      base = __shfl_sync(0xffffffffu, base, leader);
      if (key != 0xffffffffu) sorted[base + __popc(peers & ((1u << lane) - 1u))] = i | (neg ? 0x80000000u : 0u);
    } else if (key != 0xffffffffu) sorted[atomicAdd(&cursor[key], 1u)] = i | (neg ? 0x80000000u : 0u);
  });
}

// ---- 2. exclusive scan of the bucket counts over all (virtual) windows, in three launches: sums of 2048-entry tiles, a single
// CTA scanning the tile sums, and a rescan of every tile with its carry-in (a single-CTA scan of 2^19 counts cost 1 ms per MSM
// at k = 20 -- more than the sort itself).  Writes offsets and, when asked, a second copy that the scatter uses as its cursors.
constexpr uint32_t SCAN_TILE = 2048;                 // 256 threads x 8 entries
__global__ void __launch_bounds__(256) msm_tile_sum_kernel(const uint32_t* __restrict__ counts, uint32_t total, uint32_t* __restrict__ tile_sum) {
  __shared__ uint32_t wsum[8];
  const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * 8;
  uint32_t sum = 0;
#pragma unroll
  for (uint32_t j = 0; j < 8; ++j) if (base + j < total) sum += counts[base + j];
  for (uint32_t d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) { uint32_t t = 0; for (uint32_t j = 0; j < 8; ++j) t += wsum[j]; tile_sum[blockIdx.x] = t; }
}
// single CTA: exclusive scan of `total` values in place-compatible form (offsets may alias nothing of counts)
__global__ void msm_scan_kernel(const uint32_t* __restrict__ counts, uint32_t* __restrict__ offsets, uint32_t total) {
  __shared__ uint32_t part[1024];
  uint32_t tid = threadIdx.x, per = (total + blockDim.x - 1) / blockDim.x;
  uint32_t lo = min(tid * per, total), hi = min(lo + per, total), sum = 0;
  for (uint32_t j = lo; j < hi; ++j) sum += counts[j];
  part[tid] = sum;
  __syncthreads();
  for (uint32_t d = 1; d < blockDim.x; d <<= 1) {
    uint32_t v = tid >= d ? part[tid - d] : 0;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  uint32_t run = part[tid] - sum;
  for (uint32_t j = lo; j < hi; ++j) { uint32_t cnt = counts[j]; offsets[j] = run; run += cnt; }
}
__global__ void __launch_bounds__(256) msm_tile_scan_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ tile_off, uint32_t total,
                                                            uint32_t* __restrict__ offsets, uint32_t* __restrict__ cursor) {
  __shared__ uint32_t wsum[8];
  const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * 8, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t v[8], sum = 0;
#pragma unroll
  for (uint32_t j = 0; j < 8; ++j) { v[j] = base + j < total ? counts[base + j] : 0u; sum += v[j]; }
  uint32_t inc = sum;                                     // inclusive scan of the per-thread sums inside the warp
  for (uint32_t d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  uint32_t run = tile_off[blockIdx.x] + inc - sum;
  for (uint32_t j = 0; j < warp; ++j) run += wsum[j];
#pragma unroll
  for (uint32_t j = 0; j < 8; ++j)
    if (base + j < total) { offsets[base + j] = run; if (cursor) cursor[base + j] = run; run += v[j]; }
}
// tile_scratch: 2 * ceil(total / SCAN_TILE) words
static void msm_exclusive_scan(cudaStream_t st, const uint32_t* counts, uint32_t total, uint32_t* offsets, uint32_t* cursor, uint32_t* tile_scratch) {
  const uint32_t tiles = (total + SCAN_TILE - 1) / SCAN_TILE;
  msm_tile_sum_kernel<<<tiles, 256, 0, st>>>(counts, total, tile_scratch);
  msm_scan_kernel<<<1, 1024, 0, st>>>(tile_scratch, tile_scratch + tiles, tiles);
  msm_tile_scan_kernel<<<tiles, 256, 0, st>>>(counts, tile_scratch + tiles, total, offsets, cursor);
}

// ---- 4. bucket accumulation, skew-proof: every bucket's entry list is cut into segments of <= SEG
// entries; one thread per segment (so a bucket holding 30% of all points -- witness-like scalars, or the
// few-bit top window -- is spread over thousands of threads), then one thread per bucket folds its
// segment partials.
constexpr uint32_t SEG = 32;

constexpr uint32_t FOLD_SERIAL_MAX = 32;     // buckets with more segment partials than this are folded by a whole CTA
__global__ void msm_segcount_kernel(const uint32_t* __restrict__ counts, uint32_t total_buckets, uint32_t* __restrict__ nseg,
                                    uint32_t* __restrict__ large_count, uint32_t* __restrict__ large_list, uint32_t max_large) {
  uint32_t gb = blockIdx.x * blockDim.x + threadIdx.x;
  if (gb >= total_buckets) return;
  uint32_t m = (counts[gb] + SEG - 1) / SEG;
  nseg[gb] = m;
  if (m > FOLD_SERIAL_MAX) { uint32_t idx = atomicAdd(large_count, 1u); if (idx < max_large) large_list[idx] = gb; }
}
__global__ void msm_segmap_kernel(const uint32_t* __restrict__ nseg, const uint32_t* __restrict__ segoff, uint32_t total_buckets,
                                  uint32_t* __restrict__ seg_bucket) {
  uint32_t gb = blockIdx.x * blockDim.x + threadIdx.x;
  if (gb >= total_buckets) return;
  uint32_t o = segoff[gb], m = nseg[gb];
  if (m > FOLD_SERIAL_MAX) return;            // a hot bucket has thousands of segments: msm_segmap_large_kernel
  for (uint32_t j = 0; j < m; ++j) seg_bucket[o + j] = gb;
}
__global__ void msm_segmap_all_kernel(const uint32_t* __restrict__ nseg, const uint32_t* __restrict__ segoff, uint32_t total_buckets,
                                      uint32_t* __restrict__ seg_bucket) {
  uint32_t gb = blockIdx.x * blockDim.x + threadIdx.x;
  if (gb >= total_buckets) return;
  uint32_t o = segoff[gb], m = nseg[gb];
  for (uint32_t j = 0; j < m; ++j) seg_bucket[o + j] = gb;
}
__global__ void __launch_bounds__(256) msm_segmap_large_kernel(const uint32_t* __restrict__ nseg, const uint32_t* __restrict__ segoff,
                                  const uint32_t* __restrict__ large_count, const uint32_t* __restrict__ large_list, uint32_t max_large,
                                  uint32_t* __restrict__ seg_bucket) {
  const uint32_t nl = min(*large_count, max_large);
  for (uint32_t li = blockIdx.x; li < nl; li += gridDim.x) {
    const uint32_t gb = large_list[li], o = segoff[gb], m = nseg[gb];
    for (uint32_t j = threadIdx.x; j < m; j += blockDim.x) seg_bucket[o + j] = gb;
  }
}

template <class BP>
__global__ void __launch_bounds__(128, 4) msm_segment_kernel(const Affine<BP>* __restrict__ bases, const uint32_t* __restrict__ sorted,
                                  const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ counts,
                                  const uint32_t* __restrict__ nseg, const uint32_t* __restrict__ segoff,
                                  const uint32_t* __restrict__ seg_bucket, uint32_t total_buckets, uint32_t max_segs,
                                  Xyzz<BP>* __restrict__ partial) {
  uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t total_segs = segoff[total_buckets - 1] + nseg[total_buckets - 1];
  if (s >= total_segs || s >= max_segs) return;
  uint32_t gb = seg_bucket[s];
  uint32_t j0 = (s - segoff[gb]) * SEG;
  uint32_t off = offsets[gb] + j0, cnt = min(SEG, counts[gb] - j0);
  // software pipeline: the base point of entry j+1 (and the index of entry j+2) are in flight while addition j runs, so
  // the dependent  sorted[] -> bases[]  DRAM round trips overlap the ~10 field multiplications of the addition.  The point
  // in flight waits in the thread's shared-memory slot (aff_stage), not in registers: no spills instead of 60 B at 128
  // registers, 2^22 Pallas MSM 285 -> 292 M points/s on B200 (before the partial inlining of xyzz_add_mixed).
  extern __shared__ uint4 msm_stage[];
  uint4* const slot = msm_stage + threadIdx.x;
  Xyzz<BP> acc = xyzz_identity<BP>();
  const uint32_t* ent = sorted + off;
  uint32_t e = ent[0], e_n = cnt > 1 ? ent[1] : 0u;
  aff_stage<128>(slot, bases + (e & 0x7fffffffu));
  cp_async_commit();
  for (uint32_t j = 0; j < cnt; ++j) {
    const uint32_t e_nn = j + 2 < cnt ? ent[j + 2] : 0u;
    cp_async_wait<0>();
    const Affine<BP> pt = aff_staged<128, BP>(slot);       // read before the refill of the same slot is issued (same thread)
    if (j + 1 < cnt) aff_stage<128>(slot, bases + (e_n & 0x7fffffffu));
    cp_async_commit();
    xyzz_add_mixed_signed(acc, pt, (e >> 31) != 0);
    e = e_n; e_n = e_nn;
  }
  Xyzz<BP>* o = partial + s;
  fe_store(&o->x, acc.x); fe_store(&o->y, acc.y); fe_store(&o->zz, acc.zz); fe_store(&o->zzz, acc.zzz);
}

template <class BP>
__global__ void __launch_bounds__(128) msm_bucket_fold_kernel(const Xyzz<BP>* __restrict__ partial, const uint32_t* __restrict__ nseg,
                                  const uint32_t* __restrict__ segoff, uint32_t total_buckets, Xyzz<BP>* __restrict__ buckets) {
  uint32_t gb = blockIdx.x * blockDim.x + threadIdx.x;
  if (gb >= total_buckets) return;
  uint32_t o = segoff[gb], m = nseg[gb];
  if (m > FOLD_SERIAL_MAX) return;            // handled by msm_bucket_fold_large_kernel
  Xyzz<BP> acc = xyzz_identity<BP>();
  for (uint32_t j = 0; j < m; ++j) {
    const Xyzz<BP>* q = partial + o + j;
    Xyzz<BP> v; v.x = fe_load(&q->x); v.y = fe_load(&q->y); v.zz = fe_load(&q->zz); v.zzz = fe_load(&q->zzz);
    acc = (j == 0) ? v : xyzz_add(acc, v);
  }
  Xyzz<BP>* ob = buckets + gb;
  fe_store(&ob->x, acc.x); fe_store(&ob->y, acc.y); fe_store(&ob->zz, acc.zz); fe_store(&ob->zzz, acc.zzz);
}

// One CTA per oversized bucket (skewed scalars, few-bit top window): strided accumulation of its segment partials,
// then a shared-memory tree.
template <class BP>
__global__ void __launch_bounds__(256) msm_bucket_fold_large_kernel(const Xyzz<BP>* __restrict__ partial, const uint32_t* __restrict__ nseg,
                                  const uint32_t* __restrict__ segoff, const uint32_t* __restrict__ large_count,
                                  const uint32_t* __restrict__ large_list, uint32_t max_large, Xyzz<BP>* __restrict__ buckets) {
  __shared__ Xyzz<BP> sh[256];
  uint32_t nl = min(*large_count, max_large);
  for (uint32_t li = blockIdx.x; li < nl; li += gridDim.x) {
    uint32_t gb = large_list[li], o = segoff[gb], m = nseg[gb];
    Xyzz<BP> acc = xyzz_identity<BP>();
    for (uint32_t j = threadIdx.x; j < m; j += 256) {
      const Xyzz<BP>* q = partial + o + j;
      Xyzz<BP> v; v.x = fe_load(&q->x); v.y = fe_load(&q->y); v.zz = fe_load(&q->zz); v.zzz = fe_load(&q->zzz);
      acc = xyzz_add(acc, v);
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (uint32_t d = 128; d > 0; d >>= 1) {
      if (threadIdx.x < d) sh[threadIdx.x] = xyzz_add(sh[threadIdx.x], sh[threadIdx.x + d]);
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      Xyzz<BP>* ob = buckets + gb;
      fe_store(&ob->x, sh[0].x); fe_store(&ob->y, sh[0].y); fe_store(&ob->zz, sh[0].zz); fe_store(&ob->zzz, sh[0].zzz);
    }
    __syncthreads();
  }
}

template <class BP> __device__ __forceinline__ Xyzz<BP> xyzz_load(const Xyzz<BP>* p) {
  Xyzz<BP> r; r.x = fe_load(&p->x); r.y = fe_load(&p->y); r.zz = fe_load(&p->zz); r.zzz = fe_load(&p->zzz); return r;
}
template <class BP> __device__ __forceinline__ void xyzz_store(Xyzz<BP>* p, const Xyzz<BP>& v) {
  fe_store(&p->x, v.x); fe_store(&p->y, v.y); fe_store(&p->zz, v.zz); fe_store(&p->zzz, v.zzz);
}

// ---- 5. per-window reduction  R_w = sum_b (b+1) * bucket[w][b] ------------------------------------
// grid = (W, S): CTA (w, s) owns buckets [s*nb/S, (s+1)*nb/S) of window w; thread t owns a contiguous chunk:
// running sums give acc_t = sum (b - lo_t + 1) B_b and S_t = sum B_b; contribution = acc_t + lo_t * S_t.
// The S partials of a window are summed by the combine step.
template <class BP>
__global__ void __launch_bounds__(256) msm_reduce_kernel(const Xyzz<BP>* __restrict__ buckets, uint32_t nb, uint32_t splits, Xyzz<BP>* __restrict__ window_partials) {
  extern __shared__ unsigned char smem_raw[];
  Xyzz<BP>* sh = reinterpret_cast<Xyzz<BP>*>(smem_raw);
  uint32_t w = blockIdx.x, sidx = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
  uint32_t span = nb / splits, base = sidx * span;
  uint32_t per = (span + nt - 1) / nt;
  uint32_t lo = base + min(tid * per, span), hi = min(lo + per, base + span);
  Xyzz<BP> run = xyzz_identity<BP>(), acc = xyzz_identity<BP>();
  for (uint32_t b = hi; b > lo; --b) {
    Xyzz<BP> bk = xyzz_load(buckets + (size_t)w * nb + (b - 1));
    run = xyzz_add(run, bk);
    acc = xyzz_add(acc, run);
  }
  if (lo < hi && lo > 0) acc = xyzz_add(acc, xyzz_mul_u32(run, lo));
  sh[tid] = acc;
  __syncthreads();
  for (uint32_t d = nt >> 1; d > 0; d >>= 1) {
    if (tid < d) sh[tid] = xyzz_add(sh[tid], sh[tid + d]);
    __syncthreads();
  }
  if (tid == 0) xyzz_store(window_partials + (size_t)w * splits + sidx, sh[0]);
}

// sum the S partials of every window: one CTA of S threads per window, shared-memory tree (S is a power of two <= 128)
template <class BP>
__global__ void __launch_bounds__(128) msm_window_sum_kernel(const Xyzz<BP>* __restrict__ window_partials, uint32_t splits, Xyzz<BP>* __restrict__ window_sums) {
  extern __shared__ unsigned char smem_raw[];
  Xyzz<BP>* sh = reinterpret_cast<Xyzz<BP>*>(smem_raw);
  const uint32_t w = blockIdx.x, tid = threadIdx.x;
  sh[tid] = xyzz_load(window_partials + (size_t)w * splits + tid);
  __syncthreads();
  for (uint32_t d = splits >> 1; d > 0; d >>= 1) {
    if (tid < d) sh[tid] = xyzz_add(sh[tid], sh[tid + d]);
    __syncthreads();
  }
  if (tid == 0) xyzz_store(window_sums + w, sh[0]);
}

// ---- 6. Horner over windows: R = sum_w 2^(c w) R_w ; writes Jacobian (x,y,z) -----------------------
template <class BP>
__global__ void msm_combine_kernel(const Xyzz<BP>* __restrict__ window_sums, uint32_t W, uint32_t c, Jac<BP>* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  Xyzz<BP> acc = xyzz_identity<BP>();
  for (int w = (int)W - 1; w >= 0; --w) {
    for (uint32_t j = 0; j < c; ++j) acc = xyzz_dbl(acc);
    acc = xyzz_add(acc, xyzz_load(window_sums + w));
  }
  Jac<BP> j = xyzz_to_jac(acc);
  fe_store(&out->x, j.x); fe_store(&out->y, j.y); fe_store(&out->z, j.z);
}

// Jacobian -> affine, one thread per point (one inversion each; used on a handful of commitments)
template <class BP>
__global__ void jac_to_affine_kernel(const Jac<BP>* __restrict__ in, Affine<BP>* __restrict__ out, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Jac<BP> p; p.x = fe_load(&in[i].x); p.y = fe_load(&in[i].y); p.z = fe_load(&in[i].z);
  Affine<BP> r;
  if (fe_is_zero(p.z)) { r.x = fe_zero<BP>(); r.y = fe_zero<BP>(); }
  else {
    Fe<BP> zi = fe_inv_gcd(p.z), zi2 = fe_sqr(zi);
    r.x = fe_mul(p.x, zi2);
    r.y = fe_mul(p.y, fe_mul(zi2, zi));
  }
  fe_store(&out[i].x, r.x); fe_store(&out[i].y, r.y);
}

// Window size by a cost model in mixed additions: W(c) * (n + 2.8 * 2^(c-1)) -- one mixed addition per non-zero digit plus two
// full additions (14 instead of 10 multiplications each) per bucket in the running-sum reduction -- over the windows whose top
// digit is either empty or holds at least c/2 real bits of the 255-bit scalar (a top window of a few bits would pile all points
// into a handful of buckets).  A point-range shard of a large MSM (multi-GPU split) picks the window for ITS n.
static uint32_t pick_window(uint32_t n) {
  auto top_bits = [](int cc) { int W = (256 + cc - 1) / cc; return 255 - (W - 1) * cc; };
  uint32_t best = 4;
  double best_cost = 1e300;
  for (int c = 4; c <= 16; ++c) {
    const int tb = top_bits(c);
    if (c > 4 && tb > 0 && tb < c / 2) continue;
    const double W = (256 + c - 1) / c;
    const double cost = W * ((double)n + 2.8 * (double)(1u << (c - 1)));
    if (cost < best_cost) { best_cost = cost; best = (uint32_t)c; }
  }
  return best;
}

// One chunk of a batch: `n_msm` MSMs over the same `n` bases, sorted and accumulated as one problem with n_msm * W windows.
template <class BP, class SP>
static void msm_run_chunk(Ctx* ctx, const ScalarSrc<SP>& src, const Affine<BP>* bases, uint32_t n, uint32_t n_msm, uint32_t c, Jac<BP>* out) {
  cudaStream_t st = ctx->stream;
  const bzh::Field& BF = ctx->field(BP::ID);
  const uint32_t W = (256 + c - 1) / c, nb = 1u << (c - 1), WT = W * n_msm, total = WT * nb;
  const uint64_t items64 = (uint64_t)WT * n;
  BZ_CHECK(items64 < (1ull << 31) && (uint64_t)WT * nb < (1ull << 28), "msm: batch too large");
  // CTAs per window in the reduction: enough of them to fill the GPU when the batch is small, but at least 2048 buckets (8 per
  // thread) each -- every thread pays a ~25-operation scalar multiplication of its running sum on top of 2 additions per bucket,
  // so 2 buckets per thread (measured: 1.5 ms per 2^22-point MSM) lose against 8 (0.8 ms)
  uint32_t splits = 1;
  while (splits < 128 && nb / (splits * 2) >= 2048 && (uint64_t)WT * splits < 4 * 148) splits *= 2;
  const uint32_t max_segs = (uint32_t)(items64 / SEG + total);
  const uint32_t max_large = (uint32_t)(items64 / (SEG * FOLD_SERIAL_MAX) + 1);
  const uint32_t tiles = (total + SCAN_TILE - 1) / SCAN_TILE;
  ctx->scratch[0].ensure((size_t)items64 * 4);                    // point indices grouped by (MSM, window, bucket)
  ctx->scratch[2].ensure((size_t)total * 4 * 5 + (size_t)max_segs * 4 + (size_t)(max_large + 4) * 4 + (size_t)tiles * 8 + 64);
  ctx->scratch[3].ensure(((size_t)total + (size_t)WT * splits + WT + max_segs) * sizeof(Xyzz<BP>));
  uint32_t* sorted = ctx->scratch[0].as<uint32_t>();
  uint32_t* counts = ctx->scratch[2].as<uint32_t>();
  uint32_t* offsets = counts + total;
  uint32_t* nseg = offsets + total;
  uint32_t* segoff = nseg + total;
  uint32_t* cursor = segoff + total;
  uint32_t* seg_bucket = cursor + total;
  uint32_t* large_count = seg_bucket + max_segs;
  uint32_t* large_list = large_count + 4;
  uint32_t* tile_scratch = large_list + max_large;
  Xyzz<BP>* buckets = ctx->scratch[3].as<Xyzz<BP>>();
  Xyzz<BP>* wparts = buckets + total;
  Xyzz<BP>* wsums = wparts + (size_t)WT * splits;
  Xyzz<BP>* partial = wsums + WT;

  const dim3 sgrid((n + 255) / 256, n_msm);
  { ProfScope p(ctx, PROF_MSM_DIGITS);
    BZ_CUDA(cudaMemsetAsync(counts, 0, (size_t)total * 4, st));
    msm_hist_kernel<SP><<<sgrid, 256, 0, st>>>(src, n, c, W, nb, counts); }
  { ProfScope p(ctx, PROF_MSM_SORT);
    msm_exclusive_scan(st, counts, total, offsets, cursor, tile_scratch);
    msm_scatter_kernel<SP><<<sgrid, 256, 0, st>>>(src, n, c, W, nb, cursor, sorted);
    BZ_CUDA(cudaMemsetAsync(large_count, 0, 16, st));
    msm_segcount_kernel<<<(total + 255) / 256, 256, 0, st>>>(counts, total, nseg, large_count, large_list, max_large);
    msm_exclusive_scan(st, nseg, total, segoff, nullptr, tile_scratch);
    msm_segmap_kernel<<<(total + 255) / 256, 256, 0, st>>>(nseg, segoff, total, seg_bucket);
    msm_segmap_large_kernel<<<std::min<uint32_t>(max_large, 2 * 148), 256, 0, st>>>(nseg, segoff, large_count, large_list, max_large, seg_bucket); }
  { ProfScope p(ctx, PROF_MSM_BUCKET);
    msm_segment_kernel<BP><<<(max_segs + 127) / 128, 128, 128 * sizeof(Affine<BP>), st>>>(bases, sorted, offsets, counts, nseg, segoff, seg_bucket, total, max_segs, partial);
    msm_bucket_fold_kernel<BP><<<(total + 127) / 128, 128, 0, st>>>(partial, nseg, segoff, total, buckets);
    msm_bucket_fold_large_kernel<BP><<<std::min<uint32_t>(max_large, 4 * 148), 256, 0, st>>>(partial, nseg, segoff, large_count, large_list, max_large, buckets); }
  const uint32_t span = nb / splits;
  const uint32_t rthreads = span >= 256 ? 256 : (span >= 32 ? span : 32);
  { ProfScope p(ctx, PROF_MSM_REDUCE);
    msm_reduce_kernel<BP><<<dim3(WT, splits), rthreads, rthreads * sizeof(Xyzz<BP>), st>>>(buckets, nb, splits, wparts);
    msm_window_sum_kernel<BP><<<WT, splits, splits * sizeof(Xyzz<BP>), st>>>(wparts, splits, wsums); }
  ctx->kernel_launches += 16;
  BZ_CUDA(cudaGetLastError());
  // ---- Horner over the W window sums of every MSM on the host: 255 sequential doublings cost ~1.1 ms on one GPU thread and
  // ~0.1 ms on a CPU core; the data is W * 128 B per MSM, one synchronisation per chunk.
  {
    ProfScope p(ctx, PROF_MSM_COMBINE);
    std::vector<bzh::HXyzz> hw(WT);
    BZ_CUDA(cudaMemcpyAsync(hw.data(), wsums, (size_t)WT * sizeof(bzh::HXyzz), cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
    std::vector<bzh::Fe> jac(3 * (size_t)n_msm);
    for (uint32_t m = 0; m < n_msm; ++m) {
      bzh::HXyzz acc = bzh::hx_identity();
      for (int w = (int)W - 1; w >= 0; --w) {
        for (uint32_t j = 0; j < c; ++j) acc = bzh::hx_dbl(BF, acc);
        acc = bzh::hx_add(BF, acc, hw[(size_t)m * W + w]);
      }
      bzh::hx_to_jac(BF, acc, &jac[3 * (size_t)m]);
    }
    BZ_CUDA(cudaMemcpyAsync(out, jac.data(), (size_t)n_msm * 96, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaStreamSynchronize(st));
  }
}

template <class BP, class SP>
static void msm_run_t(Ctx* ctx, ScalarSrc<SP> src, const Affine<BP>* bases, uint32_t n, uint32_t n_msm, Jac<BP>* out, int c_override) {
  cudaStream_t st = ctx->stream;
  const bzh::Field& BF = ctx->field(BP::ID);
  if (n_msm == 0) return;
  if (n == 0) {
    std::vector<Jac<BP>> id(n_msm);
    memset(id.data(), 0, id.size() * sizeof(Jac<BP>));
    bzh::Fe one = BF.one();
    for (auto& j : id) memcpy(j.y.l, one.l, 32);
    BZ_CUDA(cudaMemcpyAsync(out, id.data(), id.size() * sizeof(Jac<BP>), cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaStreamSynchronize(st));
    return;
  }
  const uint32_t c = c_override > 0 ? (uint32_t)c_override : pick_window(n);
  const uint32_t W = (256 + c - 1) / c, nb = 1u << (c - 1);
  BZ_CHECK((uint64_t)W * nb <= (1u << 21), "msm: too many buckets");
  BZ_CHECK((uint64_t)W * n < (1ull << 31), "msm: n * windows too large");
  // MSMs per chunk: at most 16, and under 2^30 sorted entries / 2^24 buckets (about 4 GB of scratch at k = 20)
  uint32_t chunk = 16;
  while (chunk > 1 && ((uint64_t)chunk * W * n >= (1ull << 30) || (uint64_t)chunk * W * nb > (1ull << 24))) chunk /= 2;
  for (uint32_t m0 = 0; m0 < n_msm; m0 += chunk) {
    ScalarSrc<SP> sub = src;
    if (!sub.single) { sub.mains += m0; sub.extras += m0; }
    else BZ_CHECK(n_msm == 1, "msm: a contiguous scalar array is one MSM");
    msm_run_chunk<BP, SP>(ctx, sub, bases, n, std::min(chunk, n_msm - m0), c, out + m0);
  }
}

// curve: 0 = Vesta (scalars Fp, coordinates Fq), 1 = Pallas (scalars Fq, coordinates Fp).  All pointers device.
void msm_run(Ctx* ctx, int curve, const void* scalars, const void* bases, uint32_t n, void* out_jac, int c_override) {
  if (curve == 0) msm_run_t<FqP, FpP>(ctx, ScalarSrc<FpP>{(const Fe<FpP>*)scalars, nullptr, nullptr, 0, 0}, (const Affine<FqP>*)bases, n, 1, (Jac<FqP>*)out_jac, c_override);
  else msm_run_t<FpP, FqP>(ctx, ScalarSrc<FqP>{(const Fe<FqP>*)scalars, nullptr, nullptr, 0, 0}, (const Affine<FpP>*)bases, n, 1, (Jac<FpP>*)out_jac, c_override);
}

// A batch of MSMs over the same bases (the commitments of one round of create_proof): MSM m takes scalar g = first + i  (i < n)
// from d_main[m][g] when g < n_main, else d_extra[m][g - n_main]; `bases` is the base of point `first`.  d_main / d_extra are
// device arrays of device pointers; out_jac receives n_msm Jacobian points (96 B each).
void msm_run_batch(Ctx* ctx, int curve, const void* const* d_main, const void* const* d_extra, uint32_t n_main, uint32_t first, uint32_t n,
                   const void* bases, uint32_t n_msm, void* out_jac) {
  if (curve == 0) msm_run_t<FqP, FpP>(ctx, ScalarSrc<FpP>{nullptr, (const Fe<FpP>* const*)d_main, (const Fe<FpP>* const*)d_extra, n_main, first},
                                      (const Affine<FqP>*)bases, n, n_msm, (Jac<FqP>*)out_jac, 0);
  else msm_run_t<FpP, FqP>(ctx, ScalarSrc<FqP>{nullptr, (const Fe<FqP>* const*)d_main, (const Fe<FqP>* const*)d_extra, n_main, first},
                           (const Affine<FpP>*)bases, n, n_msm, (Jac<FpP>*)out_jac, 0);
}

// ---- shared scalars, many base sets -------------------------------------------------------------------------------------
// out[m] = sum_q s[q] * bases[q * stride + m]  for m in [0, outputs): `outputs` MSMs that share ONE scalar vector (nq scalars)
// over interleaved base sets.  This is what materialising the folded generators G' of the inner product argument needs
// (prover.cu, step 21): s = the products of the round challenges, bases = the original g.  The scalars are sorted once; the
// segment / bucket kernels take the output index as their fastest-moving thread index, so the base loads of a warp are 32
// consecutive points.  Buckets are laid out [m][window][bucket], i.e. as outputs x W virtual windows for the reduction.
template <class BP>
__global__ void __launch_bounds__(128) msm_segment_multi_kernel(const Affine<BP>* __restrict__ bases, uint32_t stride, uint32_t outputs,
                                  const uint32_t* __restrict__ sorted, const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ counts,
                                  const uint32_t* __restrict__ nseg, const uint32_t* __restrict__ segoff, const uint32_t* __restrict__ seg_bucket,
                                  uint32_t total_buckets, Xyzz<BP>* __restrict__ partial /* [segment][output] */) {
  const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y;
  const uint32_t total_segs = segoff[total_buckets - 1] + nseg[total_buckets - 1];
  if (s >= total_segs || m >= outputs) return;
  const uint32_t gb = seg_bucket[s];
  const uint32_t j0 = (s - segoff[gb]) * SEG;
  const uint32_t off = offsets[gb] + j0, cnt = min(SEG, counts[gb] - j0);
  Xyzz<BP> acc = xyzz_identity<BP>();
  for (uint32_t j = 0; j < cnt; ++j) {
    const uint32_t e = sorted[off + j];
    const Affine<BP> pt = aff_load(bases + (size_t)(e & 0x7fffffffu) * stride + m);
    xyzz_add_mixed_signed(acc, pt, (e >> 31) != 0);
  }
  xyzz_store(partial + (size_t)s * outputs + m, acc);
}
template <class BP>
__global__ void __launch_bounds__(128) msm_bucket_fold_multi_kernel(const Xyzz<BP>* __restrict__ partial, uint32_t outputs, const uint32_t* __restrict__ nseg,
                                  const uint32_t* __restrict__ segoff, uint32_t total_buckets, Xyzz<BP>* __restrict__ buckets /* [output][bucket] */) {
  const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x, gb = blockIdx.y;
  if (m >= outputs) return;
  const uint32_t o = segoff[gb], ns = nseg[gb];
  Xyzz<BP> acc = xyzz_identity<BP>();
  for (uint32_t j = 0; j < ns; ++j) {
    const Xyzz<BP> v = xyzz_load(partial + (size_t)(o + j) * outputs + m);
    acc = (j == 0) ? v : xyzz_add(acc, v);
  }
  xyzz_store(buckets + (size_t)m * total_buckets + gb, acc);
}
// Horner over the W window sums of every output, one thread per output -> Jacobian
template <class BP>
__global__ void __launch_bounds__(64) msm_combine_multi_kernel(const Xyzz<BP>* __restrict__ window_sums, uint32_t W, uint32_t c, uint32_t outputs, Jac<BP>* __restrict__ out) {
  const uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= outputs) return;
  Xyzz<BP> acc = xyzz_identity<BP>();
  for (int w = (int)W - 1; w >= 0; --w) {
    for (uint32_t j = 0; j < c; ++j) acc = xyzz_dbl(acc);
    acc = xyzz_add(acc, xyzz_load(window_sums + (size_t)m * W + w));
  }
  Jac<BP> j = xyzz_to_jac(acc);
  fe_store(&out[m].x, j.x); fe_store(&out[m].y, j.y); fe_store(&out[m].z, j.z);
}

template <class BP, class SP>
static void msm_multi_run_t(Ctx* ctx, const Fe<SP>* scalars, uint32_t nq, const Affine<BP>* bases, uint32_t stride, uint32_t outputs, Jac<BP>* out) {
  cudaStream_t st = ctx->stream;
  BZ_CHECK(nq >= 1 && outputs >= 1 && nq <= (1u << 20) && outputs <= (1u << 16), "msm (shared scalars): bad shape");
  const uint32_t c = pick_window(nq);
  const uint32_t W = (256 + c - 1) / c, nb = 1u << (c - 1), total = W * nb;
  const uint32_t items = W * nq;
  const uint32_t max_segs = items / SEG + total, max_large = items / (SEG * FOLD_SERIAL_MAX) + 1;
  const uint32_t tiles = (total + SCAN_TILE - 1) / SCAN_TILE;
  const uint64_t WT = (uint64_t)W * outputs;
  BZ_CHECK(WT * nb < (1ull << 28), "msm (shared scalars): too many buckets");
  BZ_CHECK(max_segs <= 65535 && total <= 65535, "msm (shared scalars): too many scalars for the (output, segment) grid");
  uint32_t splits = 1;                                     // the reduction sees outputs x W windows: one CTA per window fills the GPU
  ctx->scratch[0].ensure((size_t)items * 4);
  ctx->scratch[2].ensure((size_t)total * 4 * 5 + (size_t)max_segs * 4 + (size_t)(max_large + 4) * 4 + (size_t)tiles * 8 + 64);
  ctx->scratch[3].ensure(((size_t)WT * nb + WT * splits + WT + (size_t)max_segs * outputs) * sizeof(Xyzz<BP>));
  uint32_t* sorted = ctx->scratch[0].as<uint32_t>();
  uint32_t* counts = ctx->scratch[2].as<uint32_t>();
  uint32_t* offsets = counts + total;
  uint32_t* nseg = offsets + total;
  uint32_t* segoff = nseg + total;
  uint32_t* cursor = segoff + total;
  uint32_t* seg_bucket = cursor + total;
  uint32_t* large_count = seg_bucket + max_segs;
  uint32_t* large_list = large_count + 4;
  uint32_t* tile_scratch = large_list + max_large;
  Xyzz<BP>* buckets = ctx->scratch[3].as<Xyzz<BP>>();
  Xyzz<BP>* wparts = buckets + (size_t)WT * nb;
  Xyzz<BP>* wsums = wparts + (size_t)WT * splits;
  Xyzz<BP>* partial = wsums + WT;
  const ScalarSrc<SP> src{scalars, nullptr, nullptr, 0, 0};
  const dim3 sgrid((nq + 255) / 256, 1);
  { ProfScope p(ctx, PROF_MSM_SORT);
    BZ_CUDA(cudaMemsetAsync(counts, 0, (size_t)total * 4, st));
    msm_hist_kernel<SP><<<sgrid, 256, 0, st>>>(src, nq, c, W, nb, counts);
    msm_exclusive_scan(st, counts, total, offsets, cursor, tile_scratch);
    msm_scatter_kernel<SP><<<sgrid, 256, 0, st>>>(src, nq, c, W, nb, cursor, sorted);
    BZ_CUDA(cudaMemsetAsync(large_count, 0, 16, st));
    msm_segcount_kernel<<<(total + 255) / 256, 256, 0, st>>>(counts, total, nseg, large_count, large_list, max_large);
    msm_exclusive_scan(st, nseg, total, segoff, nullptr, tile_scratch);
    // every bucket's segments are written by its own thread here (a bucket of <= nq entries has few segments)
    msm_segmap_all_kernel<<<(total + 255) / 256, 256, 0, st>>>(nseg, segoff, total, seg_bucket); }
  { ProfScope p(ctx, PROF_MSM_BUCKET);
    msm_segment_multi_kernel<BP><<<dim3((outputs + 127) / 128, max_segs), 128, 0, st>>>(bases, stride, outputs, sorted, offsets, counts, nseg, segoff, seg_bucket, total, partial);
    msm_bucket_fold_multi_kernel<BP><<<dim3((outputs + 127) / 128, total), 128, 0, st>>>(partial, outputs, nseg, segoff, total, buckets); }
  const uint32_t rthreads = nb >= 256 ? 256 : (nb >= 32 ? nb : 32);
  { ProfScope p(ctx, PROF_MSM_REDUCE);
    msm_reduce_kernel<BP><<<dim3((uint32_t)WT, splits), rthreads, rthreads * sizeof(Xyzz<BP>), st>>>(buckets, nb, splits, wparts);
    msm_window_sum_kernel<BP><<<(uint32_t)WT, splits, splits * sizeof(Xyzz<BP>), st>>>(wparts, splits, wsums);
    msm_combine_multi_kernel<BP><<<(outputs + 63) / 64, 64, 0, st>>>(wsums, W, c, outputs, out); }
  ctx->kernel_launches += 16;
  BZ_CUDA(cudaGetLastError());
}

void msm_multi_run(Ctx* ctx, int curve, const void* scalars, uint32_t nq, const void* bases, uint32_t stride, uint32_t outputs, void* out_jac) {
  if (curve == 0) msm_multi_run_t<FqP, FpP>(ctx, (const Fe<FpP>*)scalars, nq, (const Affine<FqP>*)bases, stride, outputs, (Jac<FqP>*)out_jac);
  else msm_multi_run_t<FpP, FqP>(ctx, (const Fe<FqP>*)scalars, nq, (const Affine<FpP>*)bases, stride, outputs, (Jac<FpP>*)out_jac);
}

void jac_to_affine_run(Ctx* ctx, int curve, const void* jac, void* aff, uint32_t n) {
  if (!n) return;
  if (curve == 0) jac_to_affine_kernel<FqP><<<(n + 63) / 64, 64, 0, ctx->stream>>>((const Jac<FqP>*)jac, (Affine<FqP>*)aff, n);
  else jac_to_affine_kernel<FpP><<<(n + 63) / 64, 64, 0, ctx->stream>>>((const Jac<FpP>*)jac, (Affine<FpP>*)aff, n);
  ctx->kernel_launches++;
  BZ_CUDA(cudaGetLastError());
}

}  // namespace bz
