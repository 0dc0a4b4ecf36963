// 255-bit Pasta prime fields on the sm_100a integer pipe: 8 x 32-bit limbs, Montgomery form with
// R = 2^256, i.e. byte-identical to pasta_curves' in-memory [u64;4] (U: pasta_curves 0.4.1
// fields/fp.rs, fields/fq.rs; pinned at /root/reference/Cargo.lock:567-579), so `&[Fp]` crosses the
// C ABI without conversion (SURVEY §7, §8b).
//
// Both moduli are  m = 2^254 + m3*2^96 + m2*2^64 + m1*2^32 + 1  in 32-bit limbs
// [1, m1, m2, m3, 0, 0, 0, 0x40000000], and -m^-1 mod 2^32 = 0xffffffff (SURVEY App. B), so the
// Montgomery quotient digit is just q = -t0 and a reduction row costs three real multiplies.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "montmul.cuh"
#include "gcdinv.h"

namespace bz {

struct FpP {   // Pallas base field = Vesta scalar field: the NTT field and MSM-scalar field of this prover
  static constexpr int ID = 0;
  static constexpr uint32_t M1 = 0x992d30edu, M2 = 0x094cf91bu, M3 = 0x224698fcu;
  // R = 2^256 mod p, R^2, R^3 (32-bit limbs, little-endian)
  static __host__ __device__ constexpr uint32_t r1(int i) {
    constexpr uint32_t t[8] = {0xfffffffdu, 0x34786d38u, 0xe41914adu, 0x992c350bu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0x3fffffffu};
    return t[i];
  }
  static __host__ __device__ constexpr uint32_t r2(int i) {
    constexpr uint32_t t[8] = {0x0000000fu, 0x8c78ecb3u, 0x8b0de0e7u, 0xd7d30dbdu, 0xc3c95d18u, 0x7797a99bu, 0x7b9cb714u, 0x096d41afu};
    return t[i];
  }
};
struct FqP {   // Pallas scalar field = Vesta base field: coordinate field of the commitment curve
  static constexpr int ID = 1;
  static constexpr uint32_t M1 = 0x8c46eb21u, M2 = 0x0994a8ddu, M3 = 0x224698fcu;
  static __host__ __device__ constexpr uint32_t r1(int i) {
    constexpr uint32_t t[8] = {0xfffffffdu, 0x5b2b3e9cu, 0xe3420567u, 0x992c350bu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0x3fffffffu};
    return t[i];
  }
  static __host__ __device__ constexpr uint32_t r2(int i) {
    constexpr uint32_t t[8] = {0x0000000fu, 0xfc9678ffu, 0x891a16e3u, 0x67bb433du, 0x04ccf590u, 0x7fae2310u, 0x7ccfdaa9u, 0x096d41afu};
    return t[i];
  }
};

template <class P> __host__ __device__ __forceinline__ constexpr uint32_t mod_limb(int i) {
  return i == 0 ? 1u : i == 1 ? P::M1 : i == 2 ? P::M2 : i == 3 ? P::M3 : i == 7 ? 0x40000000u : 0u;
}

template <class P> struct alignas(32) Fe {
  uint32_t l[8];
};

// ---- carry-chain primitives -------------------------------------------------------------------
__device__ __forceinline__ uint32_t add_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t addc_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t addc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t sub_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t subc_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
__device__ __forceinline__ uint32_t subc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }

template <class P> __device__ __forceinline__ Fe<P> fe_zero() { Fe<P> r;
#pragma unroll
  for (int i = 0; i < 8; ++i) r.l[i] = 0; return r; }
template <class P> __device__ __forceinline__ Fe<P> fe_one() { Fe<P> r;
#pragma unroll
  for (int i = 0; i < 8; ++i) r.l[i] = P::r1(i); return r; }
template <class P> __device__ __forceinline__ Fe<P> fe_r2() { Fe<P> r;
#pragma unroll
  for (int i = 0; i < 8; ++i) r.l[i] = P::r2(i); return r; }

template <class P> __device__ __forceinline__ bool fe_is_zero(const Fe<P>& a) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) o |= a.l[i];
  return o == 0;
}
template <class P> __device__ __forceinline__ bool fe_eq(const Fe<P>& a, const Fe<P>& b) {
  uint32_t o = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) o |= a.l[i] ^ b.l[i];
  return o == 0;
}

// r = a - m if a >= m else a   (a < 2m < 2^256)
template <class P> __device__ __forceinline__ void fe_final_sub(uint32_t t[8]) {
  uint32_t u[8];
  u[0] = sub_cc(t[0], mod_limb<P>(0));
#pragma unroll
  for (int i = 1; i < 8; ++i) u[i] = subc_cc(t[i], mod_limb<P>(i));
  uint32_t borrow = subc(0u, 0u);   // 0 if no borrow, 0xffffffff if borrow
#pragma unroll
  for (int i = 0; i < 8; ++i) t[i] = borrow ? t[i] : u[i];
}

template <class P> __device__ __forceinline__ Fe<P> fe_add(const Fe<P>& a, const Fe<P>& b) {
  Fe<P> r;
  r.l[0] = add_cc(a.l[0], b.l[0]);
#pragma unroll
  for (int i = 1; i < 7; ++i) r.l[i] = addc_cc(a.l[i], b.l[i]);
  r.l[7] = addc(a.l[7], b.l[7]);      // operands < 2^255: no carry out
  fe_final_sub<P>(r.l);
  return r;
}

template <class P> __device__ __forceinline__ Fe<P> fe_sub(const Fe<P>& a, const Fe<P>& b) {
  Fe<P> r;
  r.l[0] = sub_cc(a.l[0], b.l[0]);
#pragma unroll
  for (int i = 1; i < 8; ++i) r.l[i] = subc_cc(a.l[i], b.l[i]);
  uint32_t borrow = subc(0u, 0u);
  // add back m & borrow-mask
  r.l[0] = add_cc(r.l[0], mod_limb<P>(0) & borrow);
#pragma unroll
  for (int i = 1; i < 7; ++i) r.l[i] = addc_cc(r.l[i], mod_limb<P>(i) & borrow);
  r.l[7] = addc(r.l[7], mod_limb<P>(7) & borrow);
  return r;
}

template <class P> __device__ __forceinline__ Fe<P> fe_neg(const Fe<P>& a) { return fe_sub<P>(fe_zero<P>(), a); }
template <class P> __device__ __forceinline__ Fe<P> fe_dbl(const Fe<P>& a) { return fe_add<P>(a, a); }

// Montgomery product a*b/R mod m.  Operand scanning, one reduction row per multiplier limb;
// the reduction multiplier is q = -t0 (since -m^-1 = -1 mod 2^32) and only limbs 1..3 and 7 of the
// modulus are non-trivial.  b < m required; a may be any value < 2^256 (used by from_u512).
template <class P> __device__ __forceinline__ Fe<P> fe_mul_c(const Fe<P>& a, const Fe<P>& b) {
  uint32_t t[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) t[i] = 0;
  uint32_t t8 = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    // t += a * b[i]
    uint64_t c = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      c += (uint64_t)a.l[j] * b.l[i] + t[j];
      t[j] = (uint32_t)c;
      c >>= 32;
    }
    c += t8;
    t8 = (uint32_t)c;
    uint32_t t9 = (uint32_t)(c >> 32);
    // t += q * m, then t >>= 32
    uint32_t q = 0u - t[0];
    // limb 0: t0 + q*1 = 2^32 * (t0 != 0)
    c = (t[0] != 0) ? 1ull : 0ull;
    c += (uint64_t)q * P::M1 + t[1]; t[0] = (uint32_t)c; c >>= 32;
    c += (uint64_t)q * P::M2 + t[2]; t[1] = (uint32_t)c; c >>= 32;
    c += (uint64_t)q * P::M3 + t[3]; t[2] = (uint32_t)c; c >>= 32;
    c += t[4]; t[3] = (uint32_t)c; c >>= 32;
    c += t[5]; t[4] = (uint32_t)c; c >>= 32;
    c += t[6]; t[5] = (uint32_t)c; c >>= 32;
    c += ((uint64_t)q << 30) + t[7]; t[6] = (uint32_t)c; c >>= 32;
    c += t8; t[7] = (uint32_t)c; c >>= 32;
    t8 = t9 + (uint32_t)c;
  }
  // t < 2m < 2^256  =>  t8 == 0
  fe_final_sub<P>(t);
  Fe<P> r;
#pragma unroll
  for (int i = 0; i < 8; ++i) r.l[i] = t[i];
  return r;
}

// The shipped multiplication: explicit mad.lo.cc / madc.hi.cc carry chains (montmul.cuh).  Requires a + m < 2^256
// and b < m, which every reduced operand satisfies.
// Out of line on purpose: fully inlined, the mixed-addition loop of the MSM kernel is ~180 KB of SASS and thrashes
// the 32 KB L1.5 instruction cache (ncu r1b: `no_instruction` stalls, no gain from occupancy).  One shared copy of the
// ~250-instruction multiplication keeps every hot loop inside the instruction cache.
#ifndef BZ_MUL_INLINE
#define BZ_MUL_ATTR __noinline__
#else
#define BZ_MUL_ATTR __forceinline__
#endif
template <class P> __device__ __forceinline__ void fe_mul_body(uint32_t (&r)[8], const uint32_t (&a)[8], const uint32_t (&b)[8]) {
  mm::mont_mul_wide<P::M1, P::M2, P::M3>(r, a, b);
  fe_final_sub<P>(r);
}
struct MulRet { uint4 lo, hi; };      // returned in registers by the device ABI
template <class P> __device__ BZ_MUL_ATTR MulRet fe_mul_raw(uint4 a0, uint4 a1, uint4 b0, uint4 b1) {
  uint32_t a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
  uint32_t b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
  uint32_t r[8];
  fe_mul_body<P>(r, a, b);
  MulRet o;
  o.lo = make_uint4(r[0], r[1], r[2], r[3]); o.hi = make_uint4(r[4], r[5], r[6], r[7]);
  return o;
}
template <class P> __device__ __forceinline__ Fe<P> fe_mul(const Fe<P>& a, const Fe<P>& b) {
  MulRet o = fe_mul_raw<P>(make_uint4(a.l[0], a.l[1], a.l[2], a.l[3]), make_uint4(a.l[4], a.l[5], a.l[6], a.l[7]),
                           make_uint4(b.l[0], b.l[1], b.l[2], b.l[3]), make_uint4(b.l[4], b.l[5], b.l[6], b.l[7]));
  Fe<P> r;
  r.l[0] = o.lo.x; r.l[1] = o.lo.y; r.l[2] = o.lo.z; r.l[3] = o.lo.w;
  r.l[4] = o.hi.x; r.l[5] = o.hi.y; r.l[6] = o.hi.z; r.l[7] = o.hi.w;
  return r;
}

// The same product inlined at the call site, for the few hot call sites where the operand / result moves of the call (~22
// fma-pipe instructions per multiplication) cost more than the instruction-cache space (see xyzz_add_mixed).
template <class P> __device__ __forceinline__ Fe<P> fe_mul_inline(const Fe<P>& a, const Fe<P>& b) {
  Fe<P> r;
  fe_mul_body<P>(r.l, a.l, b.l);
  return r;
}

template <class P> __device__ __forceinline__ Fe<P> fe_sqr(const Fe<P>& a) { return fe_mul<P>(a, a); }

// Montgomery <-> canonical
template <class P> __device__ __forceinline__ Fe<P> fe_to_mont(const Fe<P>& a) { return fe_mul<P>(a, fe_r2<P>()); }
template <class P> __device__ __forceinline__ Fe<P> fe_from_mont(const Fe<P>& a) {
  Fe<P> one = fe_zero<P>(); one.l[0] = 1;
  return fe_mul<P>(a, one);
}
template <class P> __device__ __forceinline__ Fe<P> fe_from_u32(uint32_t v) {
  Fe<P> a = fe_zero<P>(); a.l[0] = v;
  return fe_to_mont<P>(a);
}

// a^e for a 256-bit exponent given as 8 limbs (uniform across the warp in all our uses)
template <class P> __device__ __noinline__ Fe<P> fe_pow(const Fe<P>& a, const uint32_t e[8]) {
  Fe<P> acc = fe_one<P>();
  for (int i = 255; i >= 0; --i) {
    acc = fe_sqr<P>(acc);
    if ((e[i >> 5] >> (i & 31)) & 1) acc = fe_mul<P>(acc, a);
  }
  return acc;
}
template <class P> __device__ __forceinline__ Fe<P> fe_pow_u64(const Fe<P>& a, uint64_t e) {
  Fe<P> acc = fe_one<P>();
  bool started = false;
  for (int i = 63; i >= 0; --i) {
    if (started) acc = fe_sqr<P>(acc);
    if ((e >> i) & 1) { acc = started ? fe_mul<P>(acc, a) : a; started = true; }
  }
  return acc;
}
// Fermat inverse (0 -> 0)
template <class P> __device__ __noinline__ Fe<P> fe_inv(const Fe<P>& a) {
  uint32_t e[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) e[i] = mod_limb<P>(i);
  e[0] = 0xffffffffu;   // m - 2: limb0 is 1 -> borrow through: (m1..): 1 - 2 = -1 mod 2^32 with borrow from limb 1
  e[1] = P::M1 - 1u;
  return fe_pow<P>(a, e);
}

// Inversion by the binary GCD of gcdinv.h (0 -> 0):  (aR)^-1 = a^-1 R^-1, and two Montgomery multiplications by R^2 give a^-1 R.
// ALU-pipe work instead of a Fermat chain on the fma pipe (data-dependent loops: meant for single-lane, latency-bound call sites).
template <class P> __device__ __noinline__ Fe<P> fe_inv_gcd(const Fe<P>& a) {
  uint32_t p[8], r[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) p[i] = mod_limb<P>(i);
  gcdinv::inverse(r, a.l, p);
  Fe<P> x;
#pragma unroll
  for (int i = 0; i < 8; ++i) x.l[i] = r[i];
  return fe_to_mont<P>(fe_to_mont<P>(x));
}

// 256-bit vector load/store of one element (sm_100a has 256-bit global accesses; two 128-bit halves
// are emitted where the compiler prefers)
template <class P> __device__ __forceinline__ Fe<P> fe_load(const Fe<P>* p) {
  Fe<P> r;
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
  r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
  return r;
}
template <class P> __device__ __forceinline__ void fe_store(Fe<P>* p, const Fe<P>& v) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
  q[1] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

// pasta `from_u512`: (lo + hi * 2^256) mod m, as Montgomery: lo*R2/R + hi*R3/R, with R3 = R2*R2/R
template <class P> __device__ __forceinline__ Fe<P> fe_from_u512(const uint32_t w[16]) {
  Fe<P> lo, hi;
#pragma unroll
  for (int i = 0; i < 8; ++i) { lo.l[i] = w[i]; hi.l[i] = w[8 + i]; }
  Fe<P> r2 = fe_r2<P>();
  Fe<P> r3 = fe_mul<P>(r2, r2);
  return fe_add<P>(fe_mul_c<P>(lo, r2), fe_mul_c<P>(hi, r3));     // lo / hi are arbitrary 256-bit values
}

using Fp = Fe<FpP>;
using Fq = Fe<FqP>;

}  // namespace bz
