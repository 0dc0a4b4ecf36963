#pragma once
#include "common.h"
namespace bz {
struct FixedBase {
  int curve = 0;
  uint32_t npts = 0, c = 0, W = 0, nbk = 0;
  DevBuf table;     // Affine[W][nbk][npts]
};
void fixed_base_build(Ctx* ctx, FixedBase& fb, int curve, const void* bases_dev, uint32_t npts, uint32_t c);
// d_main / d_extra: DEVICE arrays of n_msm device pointers (extra may be null); out: n_msm affine points (device, 64 B
// each), or -- xyzz_out -- the unnormalised XYZZ sums (128 B each: X, Y, ZZ, ZZZ) for callers that normalise on the host
// (one batched inversion there beats a single-thread Fermat chain per commitment on the device)
void fixed_msm_run(Ctx* ctx, const FixedBase& fb, const void* const* d_main, uint32_t n_main, const void* const* d_extra,
                   uint32_t n_msm, void* d_out, bool xyzz_out = false);
}  // namespace bz
