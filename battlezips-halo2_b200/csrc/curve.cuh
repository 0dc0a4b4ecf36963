// Pasta curves y^2 = x^3 + 5 on the device (U: pasta_curves 0.4.1 curves.rs; SURVEY §8 a12).
// ABI layouts: affine = x||y (64 B, Montgomery, identity = all zero), Jacobian = x||y||z (96 B,
// identity z = 0).  Accumulation inside kernels uses extended Jacobian "XYZZ" coordinates
// (x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2): mixed addition 8M+2S and no inversion anywhere.
// Group results are only ever compared/serialised after to_affine, so any representative of the
// projective class is bit-exact with the reference (SURVEY §0 fact 5).
#pragma once
#include "field.cuh"

namespace bz {

template <class BP> struct Affine { Fe<BP> x, y; };
template <class BP> struct Jac { Fe<BP> x, y, z; };
template <class BP> struct Xyzz { Fe<BP> x, y, zz, zzz; };

template <class BP> __device__ __forceinline__ bool aff_is_identity(const Affine<BP>& a) { return fe_is_zero(a.x) && fe_is_zero(a.y); }
template <class BP> __device__ __forceinline__ bool xyzz_is_identity(const Xyzz<BP>& a) { return fe_is_zero(a.zz); }

template <class BP> __device__ __forceinline__ Xyzz<BP> xyzz_identity() {
  Xyzz<BP> r; r.x = fe_zero<BP>(); r.y = fe_zero<BP>(); r.zz = fe_zero<BP>(); r.zzz = fe_zero<BP>(); return r;
}
template <class BP> __device__ __forceinline__ Xyzz<BP> xyzz_from_affine(const Affine<BP>& a) {
  Xyzz<BP> r;
  if (aff_is_identity(a)) return xyzz_identity<BP>();
  r.x = a.x; r.y = a.y; r.zz = fe_one<BP>(); r.zzz = fe_one<BP>();
  return r;
}

// dbl-2008-s-1 for a = 0
template <class BP> __device__ __noinline__ Xyzz<BP> xyzz_dbl(const Xyzz<BP>& p) {
  if (xyzz_is_identity(p)) return p;
  Fe<BP> u = fe_dbl(p.y);
  Fe<BP> v = fe_sqr(u);
  Fe<BP> w = fe_mul(u, v);
  Fe<BP> s = fe_mul(p.x, v);
  Fe<BP> xx = fe_sqr(p.x);
  Fe<BP> m = fe_add(fe_dbl(xx), xx);
  Xyzz<BP> r;
  r.x = fe_sub(fe_sqr(m), fe_dbl(s));
  r.y = fe_sub(fe_mul(m, fe_sub(s, r.x)), fe_mul(w, p.y));
  r.zz = fe_mul(v, p.zz);
  r.zzz = fe_mul(w, p.zzz);
  return r;
}

// mixed addition acc += q (affine), complete: handles identity / doubling / inverse (madd-2008-s).
// The loop body of both MSM accumulation kernels.  Six of its ten multiplications are inlined, four stay calls of the
// shared out-of-line fe_mul: measured on B200 (1000 W), table-MSM accumulation per IPA-round launch at k = 11, c = 16
// (scripts/fb_accumulate_time.py): 0 / 2 / 4 / 6 / 7 / 8 / 10 inlined 0.358 / 0.349 / 0.343 / 0.335 / 0.337 / 0.343 /
// 0.346 ms -- every inlined product drops the call's operand and result moves, until the loop outgrows the instruction
// cache.
template <class BP> __device__ __forceinline__ void xyzz_add_mixed(Xyzz<BP>& acc, const Affine<BP>& q) {
  if (aff_is_identity(q)) return;
  if (xyzz_is_identity(acc)) { acc = xyzz_from_affine(q); return; }
  Fe<BP> u2 = fe_mul_inline(q.x, acc.zz);
  Fe<BP> s2 = fe_mul_inline(q.y, acc.zzz);
  Fe<BP> p = fe_sub(u2, acc.x);
  Fe<BP> r = fe_sub(s2, acc.y);
  if (fe_is_zero(p)) {
    if (fe_is_zero(r)) { acc = xyzz_dbl(xyzz_from_affine(q)); }
    else acc = xyzz_identity<BP>();
    return;
  }
  Fe<BP> pp = fe_sqr(p);
  Fe<BP> ppp = fe_mul_inline(p, pp);
  Fe<BP> qq = fe_mul_inline(acc.x, pp);
  Fe<BP> x3 = fe_sub(fe_sub(fe_sqr(r), ppp), fe_dbl(qq));
  acc.y = fe_sub(fe_mul(r, fe_sub(qq, x3)), fe_mul(acc.y, ppp));
  acc.x = x3;
  acc.zz = fe_mul_inline(acc.zz, pp);
  acc.zzz = fe_mul_inline(acc.zzz, ppp);
}

// acc += sign ? -q : q
template <class BP> __device__ __forceinline__ void xyzz_add_mixed_signed(Xyzz<BP>& acc, Affine<BP> q, bool negate) {
  if (negate) q.y = fe_neg(q.y);    // identity (0,0) stays (0,0)
  xyzz_add_mixed(acc, q);
}

// full addition (add-2008-s), complete
template <class BP> __device__ __noinline__ Xyzz<BP> xyzz_add(const Xyzz<BP>& a, const Xyzz<BP>& b) {
  if (xyzz_is_identity(a)) return b;
  if (xyzz_is_identity(b)) return a;
  Fe<BP> u1 = fe_mul(a.x, b.zz);
  Fe<BP> u2 = fe_mul(b.x, a.zz);
  Fe<BP> s1 = fe_mul(a.y, b.zzz);
  Fe<BP> s2 = fe_mul(b.y, a.zzz);
  Fe<BP> p = fe_sub(u2, u1);
  Fe<BP> r = fe_sub(s2, s1);
  if (fe_is_zero(p)) {
    if (fe_is_zero(r)) return xyzz_dbl(a);
    return xyzz_identity<BP>();
  }
  Fe<BP> pp = fe_sqr(p);
  Fe<BP> ppp = fe_mul(p, pp);
  Fe<BP> qq = fe_mul(u1, pp);
  Xyzz<BP> o;
  o.x = fe_sub(fe_sub(fe_sqr(r), ppp), fe_dbl(qq));
  o.y = fe_sub(fe_mul(r, fe_sub(qq, o.x)), fe_mul(s1, ppp));
  o.zz = fe_mul(fe_mul(a.zz, b.zz), pp);
  o.zzz = fe_mul(fe_mul(a.zzz, b.zzz), ppp);
  return o;
}

template <class BP> __device__ __forceinline__ Xyzz<BP> xyzz_neg(const Xyzz<BP>& a) {
  Xyzz<BP> r = a; r.y = fe_neg(a.y); return r;
}

// XYZZ -> Jacobian without inversion: Z = ZZZ (= z^3)  =>  X' = X*ZZ^2, Y' = Y*ZZZ^2
template <class BP> __device__ __forceinline__ Jac<BP> xyzz_to_jac(const Xyzz<BP>& a) {
  Jac<BP> r;
  if (xyzz_is_identity(a)) { r.x = fe_zero<BP>(); r.y = fe_one<BP>(); r.z = fe_zero<BP>(); return r; }
  r.x = fe_mul(a.x, fe_sqr(a.zz));
  r.y = fe_mul(a.y, fe_sqr(a.zzz));
  r.z = a.zzz;
  return r;
}
template <class BP> __device__ __forceinline__ Xyzz<BP> jac_to_xyzz(const Jac<BP>& a) {
  Xyzz<BP> r;
  if (fe_is_zero(a.z)) return xyzz_identity<BP>();
  r.x = a.x; r.y = a.y; r.zz = fe_sqr(a.z); r.zzz = fe_mul(r.zz, a.z);
  return r;
}
// one inversion
template <class BP> __device__ __forceinline__ Affine<BP> xyzz_to_affine(const Xyzz<BP>& a) {
  Affine<BP> r;
  if (xyzz_is_identity(a)) { r.x = fe_zero<BP>(); r.y = fe_zero<BP>(); return r; }
  Fe<BP> zi = fe_inv_gcd(a.zzz);             // 1/z^3 (binary GCD: the callers run this on one lane per point)
  Fe<BP> zi2 = fe_mul(fe_sqr(zi), a.zz);     // z^-6 * z^2 ... = z^-4? no: see below
  // zz = z^2, zzz = z^3: 1/zz = zzz^-2 * zz^2 = z^-6 * z^4 = z^-2
  zi2 = fe_mul(zi2, a.zz);
  r.x = fe_mul(a.x, zi2);
  r.y = fe_mul(a.y, zi);
  return r;
}

// scalar multiple by a small non-negative integer (used by bucket-reduction chunk combine)
template <class BP> __device__ __noinline__ Xyzz<BP> xyzz_mul_u32(const Xyzz<BP>& p, uint32_t k) {
  Xyzz<BP> acc = xyzz_identity<BP>();
  for (int i = 31; i >= 0; --i) {
    acc = xyzz_dbl(acc);
    if ((k >> i) & 1) acc = xyzz_add(acc, p);
  }
  return acc;
}

// [k]P, k canonical 256-bit, double-and-add from the top bit
template <class BP> __device__ Xyzz<BP> xyzz_mul_scalar(const Xyzz<BP>& p, const uint32_t k[8]) {
  Xyzz<BP> acc = xyzz_identity<BP>();
  int top = 255;
  while (top >= 0 && !((k[top >> 5] >> (top & 31)) & 1)) --top;
  for (int i = top; i >= 0; --i) {
    acc = xyzz_dbl(acc);
    if ((k[i >> 5] >> (i & 31)) & 1) acc = xyzz_add(acc, p);
  }
  return acc;
}

template <class BP> __device__ __forceinline__ Affine<BP> aff_load(const Affine<BP>* p) {
  Affine<BP> r; r.x = fe_load(&p->x); r.y = fe_load(&p->y); return r;
}

// Gather staging of the accumulation loops (fixedmsm.cu, msm.cu): the affine point a thread adds next is copied into the
// thread's own shared-memory slot by cp.async (4 x 16 B, L1-allocating .ca, like the register loads it replaces) instead
// of waiting in 16 registers while the current addition runs.  Chunk k of the slot of thread t is uint4 k * THREADS + t
// of the slot array: a warp's copies and reads of one chunk are 512 contiguous bytes (no bank conflicts).
__device__ __forceinline__ void cp_async16_ca(uint4* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" :: "r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" :: "n"(N) : "memory"); }

template <int THREADS, class BP> __device__ __forceinline__ void aff_stage(uint4* slot, const Affine<BP>* src) {
  const uint4* g = reinterpret_cast<const uint4*>(src);
#pragma unroll
  for (int k = 0; k < 4; ++k) cp_async16_ca(slot + k * THREADS, g + k);
}
template <int THREADS, class BP> __device__ __forceinline__ Affine<BP> aff_staged(const uint4* slot) {
  Affine<BP> r;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint4 v = slot[k * THREADS];
    Fe<BP>& f = k < 2 ? r.x : r.y;
    const int o = (k & 1) * 4;
    f.l[o] = v.x; f.l[o + 1] = v.y; f.l[o + 2] = v.z; f.l[o + 3] = v.w;
  }
  return r;
}

}  // namespace bz
