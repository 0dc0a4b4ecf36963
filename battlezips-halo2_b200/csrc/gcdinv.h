// Modular inversion by the binary extended Euclidean algorithm on 8 x 32-bit limbs, for moduli with p = 1 (mod 2^32)
// (both Pasta primes; field.cuh `mod_limb`).  Groundwork for round 2: `fe_inv` is a Fermat chain of ~320 DEPENDENT field
// multiplications (~77 K instructions, half of them on the fma-heavy pipe every kernel of this library is bound by, and
// 130 - 180 us of latency on a lone warp); this routine needs ~30 K instructions, practically all of them on the ALU pipe
// (which sits at ~33 %), so the inversions inside the grand-product finish, the batch-inversion kernels and the table build
// stop competing with the multiplications.  Used through `fe_inv_gcd`
// (field.cuh) wherever ONE lane inverts while the rest of its warp waits: the grand-product finish, XYZZ / Jacobian ->
// affine, and `bz_field_op` op 9.  Checked on the CPU (tests/test_gcdinv_host.py runs this very code, compiled for the
// host, against big-integer inverses) and on the device against the Fermat chain and the oracle
// (tests/test_gpu_arith.py::test_binary_gcd_inverse_on_device, green on B200 in round 2).
//
// Invariants:  b * a = u  and  c * a = v  (mod p), u and v odd after the shifts; gcd(u, v) = 1, so the loop ends with
// u = v = 1 and b = a^-1.  Trailing zeros are removed all at once: because p = 1 (mod 2^32), p^-1 = 1 (mod 2^k) for k <= 32,
// hence  b / 2^k = (b + m p) >> k  with  m = -b mod 2^k.
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define BZ_HD __host__ __device__ __forceinline__
#else
#define BZ_HD inline
#endif

namespace bz {
namespace gcdinv {

BZ_HD int ctz32(uint32_t x) {
#ifdef __CUDA_ARCH__
  return __ffs((int)x) - 1;
#else
  return __builtin_ctz(x);
#endif
}
BZ_HD int cmp(const uint32_t (&x)[8], const uint32_t (&y)[8]) {      // -1, 0, +1
  for (int i = 7; i >= 0; --i) {
    if (x[i] != y[i]) return x[i] > y[i] ? 1 : -1;
  }
  return 0;
}
BZ_HD void sub(uint32_t (&x)[8], const uint32_t (&y)[8]) {           // x -= y  (x >= y)
  uint64_t borrow = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint64_t d = (uint64_t)x[i] - y[i] - borrow;
    x[i] = (uint32_t)d;
    borrow = (d >> 32) & 1u;
  }
}
BZ_HD void submod(uint32_t (&x)[8], const uint32_t (&y)[8], const uint32_t (&p)[8]) {   // x = x - y mod p  (x, y < p)
  uint64_t borrow = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint64_t d = (uint64_t)x[i] - y[i] - borrow;
    x[i] = (uint32_t)d;
    borrow = (d >> 32) & 1u;
  }
  if (borrow) {
    uint64_t carry = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint64_t s = (uint64_t)x[i] + p[i] + carry;
      x[i] = (uint32_t)s;
      carry = s >> 32;
    }
  }
}
BZ_HD void shr(uint32_t (&x)[8], int k) {                              // x >>= k, 1 <= k <= 31
#pragma unroll
  for (int i = 0; i < 7; ++i) x[i] = (x[i] >> k) | (x[i + 1] << (32 - k));
  x[7] >>= k;
}
// x = x / 2^k mod p, 1 <= k <= 31, x < p, p = 1 (mod 2^32)
BZ_HD void div2k(uint32_t (&x)[8], int k, const uint32_t (&p)[8]) {
  const uint32_t m = (0u - x[0]) & ((1u << k) - 1u);
  uint32_t t[9];
  uint64_t carry = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint64_t s = (uint64_t)m * p[i] + x[i] + carry;
    t[i] = (uint32_t)s;
    carry = s >> 32;
  }
  t[8] = (uint32_t)carry;
#pragma unroll
  for (int i = 0; i < 8; ++i) x[i] = (t[i] >> k) | (t[i + 1] << (32 - k));
}

// out = a^-1 mod p for 0 < a < p (p prime, p = 1 mod 2^32); out = 0 for a = 0 (ff's convention for BatchInvert)
BZ_HD void inverse(uint32_t (&out)[8], const uint32_t (&a)[8], const uint32_t (&p)[8]) {
  uint32_t u[8], v[8], b[8], c[8];
  uint32_t any = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) { u[i] = a[i]; v[i] = p[i]; b[i] = 0; c[i] = 0; any |= a[i]; }
  if (!any) {
#pragma unroll
    for (int i = 0; i < 8; ++i) out[i] = 0;
    return;
  }
  b[0] = 1;
  for (;;) {
    while (!(u[0] & 1u)) { const int k = u[0] ? ctz32(u[0]) : 31; shr(u, k); div2k(b, k, p); }
    while (!(v[0] & 1u)) { const int k = v[0] ? ctz32(v[0]) : 31; shr(v, k); div2k(c, k, p); }
    const int s = cmp(u, v);
    if (s == 0) break;
    if (s > 0) { sub(u, v); submod(b, c, p); }
    else { sub(v, u); submod(c, b, p); }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) out[i] = b[i];
}

}  // namespace gcdinv
}  // namespace bz
