// extern "C" surface of libbzhalo2 (declared in include/bzhalo2.h).
#include "../../include/bzhalo2.h"
#include "common.h"
#include <set>

namespace bz {
void msm_run(Ctx* ctx, int curve, const void* scalars, const void* bases, uint32_t n, void* out_jac, int c_override);
void jac_to_affine_run(Ctx* ctx, int curve, const void* jac, void* aff, uint32_t n);
void jac_sum_run(Ctx* ctx, int curve, const void* d_jac, uint32_t count, void* d_out_affine);
void field_op_run(Ctx* ctx, int field, int op, const void* a, const void* b, void* out, uint64_t n);
void curve_op_run(Ctx* ctx, int curve, int op, const void* a, const void* b, void* out, uint64_t n);
void batch_invert_assigned_run(Ctx* ctx, int field, const void* num, const void* den, void* out, uint64_t n);

Ctx::~Ctx() {}
}  // namespace bz


#define BZ_TRY(ctx_, ...)                                    \
  if (!(ctx_)) return BZ_ERR_INVALID;                        \
  try {                                                      \
    cudaSetDevice((ctx_)->c.device);                         \
    __VA_ARGS__;                                             \
    return BZ_OK;                                            \
  } catch (const bz::Error& e) {                             \
    (ctx_)->c.last_error = e.what();                         \
    return e.code;                                           \
  } catch (const std::exception& e) {                        \
    (ctx_)->c.last_error = e.what();                         \
    return BZ_ERR_INVALID;                                   \
  }

extern "C" {

__attribute__((visibility("default"))) const char* bz_version(void) { return "bzhalo2-b200 0.1 (sm_100a)"; }

__attribute__((visibility("default"))) int bz_ctx_create(int device, void* stream, bz_ctx** out) {
  if (!out) return BZ_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return BZ_ERR_CUDA;   // no CPU fallback
  if (cudaSetDevice(device) != cudaSuccess) return BZ_ERR_CUDA;
  bz_ctx* h = new (std::nothrow) bz_ctx();
  if (!h) return BZ_ERR_INVALID;
  h->c.device = device;
  if (stream) h->c.stream = (cudaStream_t)stream;
  else {
    if (cudaStreamCreateWithFlags(&h->c.stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return BZ_ERR_CUDA; }
    h->own_stream = true;
  }
  cudaDeviceGetAttribute(&h->c.sm_count, cudaDevAttrMultiProcessorCount, device);
  *out = h;
  return BZ_OK;
}

__attribute__((visibility("default"))) void bz_ctx_destroy(bz_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->c.device);
  cudaStreamSynchronize(ctx->c.stream);
  for (void* p : ctx->allocs) cudaFree(p);
  if (ctx->own_stream) cudaStreamDestroy(ctx->c.stream);
  delete ctx;
}

__attribute__((visibility("default"))) int bz_ctx_set_sharding(bz_ctx* ctx, uint32_t rank, uint32_t world, void* d_send, void* d_recv, size_t capacity_per_rank,
                                                               bz_allgather_fn exchange, void* user) {
  BZ_TRY(ctx, {
    BZ_CHECK(world >= 1 && rank < world, "bad rank / world");
    BZ_CHECK(world == 1 || (d_send && d_recv && exchange && capacity_per_rank >= 96), "sharding needs exchange buffers and a callback");
    bz::Ctx& c = ctx->c;
    c.shard_rank = rank; c.shard_world = world; c.shard_send = d_send; c.shard_recv = d_recv; c.shard_cap = capacity_per_rank;
    c.shard_exchange = exchange; c.shard_user = user;
  });
}

__attribute__((visibility("default"))) const char* bz_last_error(bz_ctx* ctx) { return ctx ? ctx->c.last_error.c_str() : "null context"; }
__attribute__((visibility("default"))) uint64_t bz_kernel_launches(bz_ctx* ctx) { return ctx ? ctx->c.kernel_launches : 0; }

__attribute__((visibility("default"))) int bz_sync(bz_ctx* ctx) { BZ_TRY(ctx, BZ_CUDA(cudaStreamSynchronize(ctx->c.stream))); }

__attribute__((visibility("default"))) int bz_dev_alloc(bz_ctx* ctx, size_t bytes, void** dptr) {
  BZ_TRY(ctx, {
    BZ_CHECK(dptr, "null out pointer");
    BZ_CUDA(cudaMalloc(dptr, bytes ? bytes : 1));
    ctx->allocs.insert(*dptr);
  });
}
__attribute__((visibility("default"))) int bz_dev_free(bz_ctx* ctx, void* dptr) {
  BZ_TRY(ctx, {
    BZ_CHECK(ctx->allocs.erase(dptr) == 1, "bz_dev_free: pointer not owned by this context");
    BZ_CUDA(cudaStreamSynchronize(ctx->c.stream));
    BZ_CUDA(cudaFree(dptr));
  });
}
__attribute__((visibility("default"))) int bz_h2d(bz_ctx* ctx, void* dptr, const void* host, size_t bytes) {
  BZ_TRY(ctx, BZ_CUDA(cudaMemcpyAsync(dptr, host, bytes, cudaMemcpyHostToDevice, ctx->c.stream)));
}
__attribute__((visibility("default"))) int bz_d2h(bz_ctx* ctx, void* host, const void* dptr, size_t bytes) {
  BZ_TRY(ctx, {
    BZ_CUDA(cudaMemcpyAsync(host, dptr, bytes, cudaMemcpyDeviceToHost, ctx->c.stream));
    BZ_CUDA(cudaStreamSynchronize(ctx->c.stream));
  });
}

// ---- per-kernel-class device timing ------------------------------------------------------------------
static void prof_drain(bz_ctx* ctx) {
  cudaStreamSynchronize(ctx->c.stream);
  for (auto& r : ctx->c.prof) {
    float ms = 0; cudaEventElapsedTime(&ms, r.a, r.b);
    ctx->c.prof_ms[r.tag] += ms; ctx->c.prof_count[r.tag]++;
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  ctx->c.prof.clear();
}
__attribute__((visibility("default"))) int bz_profile_enable(bz_ctx* ctx, int on) {
  BZ_TRY(ctx, {
    prof_drain(ctx);
    ctx->c.profiling = on != 0;
    for (int i = 0; i < bz::PROF_NTAGS; ++i) { ctx->c.prof_ms[i] = 0; ctx->c.prof_count[i] = 0; }
  });
}
__attribute__((visibility("default"))) int bz_profile_read(bz_ctx* ctx, int tag, double* total_ms, uint64_t* count) {
  BZ_TRY(ctx, {
    BZ_CHECK(tag >= 0 && tag < bz::PROF_NTAGS, "bad profile tag");
    prof_drain(ctx);
    if (total_ms) *total_ms = ctx->c.prof_ms[tag];
    if (count) *count = ctx->c.prof_count[tag];
  });
}

__attribute__((visibility("default"))) int bz_profile_counter(bz_ctx* ctx, int which, uint64_t* value, int reset) {
  BZ_TRY(ctx, {
    BZ_CHECK(which >= 0 && which < 8 && value, "bad counter");
    *value = 0;
    if (ctx->c.counters.p) {
      BZ_CUDA(cudaMemcpyAsync(value, (uint64_t*)ctx->c.counters.p + which, 8, cudaMemcpyDeviceToHost, ctx->c.stream));
      BZ_CUDA(cudaStreamSynchronize(ctx->c.stream));
      if (reset) BZ_CUDA(cudaMemsetAsync((uint64_t*)ctx->c.counters.p + which, 0, 8, ctx->c.stream));
    }
  });
}

// Integer-pipe peak: independent 32-bit multiply-add chains on every SM; returns IMAD/s (the denominator for
// the MSM / quotient integer roofline; SURVEY §8d "must be measured").
__global__ void imad_peak_kernel(uint32_t* out, uint32_t iters) {
  uint32_t a0 = threadIdx.x + 1, a1 = a0 * 3, a2 = a0 * 5, a3 = a0 * 7, a4 = a0 * 11, a5 = a0 * 13, a6 = a0 * 17, a7 = a0 * 19;
  const uint32_t m = blockIdx.x * 2 + 1, c = 0x9e3779b9u;
  for (uint32_t i = 0; i < iters; ++i) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      a0 = a0 * m + c; a1 = a1 * m + c; a2 = a2 * m + c; a3 = a3 * m + c;
      a4 = a4 * m + c; a5 = a5 * m + c; a6 = a6 * m + c; a7 = a7 * m + c;
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}
// same, with 32x32+64 -> 64 multiply-adds (IMAD.WIDE.U32), the instruction the Montgomery multiplication is made of
__global__ void imad_wide_peak_kernel(unsigned long long* out, uint32_t iters) {
  unsigned long long a0 = threadIdx.x + 1, a1 = a0 * 3, a2 = a0 * 5, a3 = a0 * 7, a4 = a0 * 11, a5 = a0 * 13, a6 = a0 * 17, a7 = a0 * 19;
  const uint32_t m = blockIdx.x * 2 + 1;
  for (uint32_t i = 0; i < iters; ++i) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      a0 = (unsigned long long)(uint32_t)a0 * m + a0; a1 = (unsigned long long)(uint32_t)a1 * m + a1;
      a2 = (unsigned long long)(uint32_t)a2 * m + a2; a3 = (unsigned long long)(uint32_t)a3 * m + a3;
      a4 = (unsigned long long)(uint32_t)a4 * m + a4; a5 = (unsigned long long)(uint32_t)a5 * m + a5;
      a6 = (unsigned long long)(uint32_t)a6 * m + a6; a7 = (unsigned long long)(uint32_t)a7 * m + a7;
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}
// FP64 pipe probes for the round-2 question "can a 52-bit-limb DFMA multiplier run beside the IMAD one?":
// mode 2 = DFMA chains only, mode 3 = IMAD.WIDE and DFMA chains interleaved in the same warp (ops counted together)
__global__ void dfma_peak_kernel(double* out, uint32_t iters, int mixed) {
  double d0 = threadIdx.x + 1.0, d1 = d0 * 3, d2 = d0 * 5, d3 = d0 * 7, d4 = d0 * 11, d5 = d0 * 13, d6 = d0 * 17, d7 = d0 * 19;
  const double m = 1.0000001 + blockIdx.x * 1e-9, c = 0.5;
  unsigned long long a0 = threadIdx.x + 1, a1 = a0 * 3, a2 = a0 * 5, a3 = a0 * 7, a4 = a0 * 11, a5 = a0 * 13, a6 = a0 * 17, a7 = a0 * 19;
  const uint32_t mi = blockIdx.x * 2 + 1;
  for (uint32_t i = 0; i < iters; ++i) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      d0 = fma(d0, m, c); d1 = fma(d1, m, c); d2 = fma(d2, m, c); d3 = fma(d3, m, c);
      d4 = fma(d4, m, c); d5 = fma(d5, m, c); d6 = fma(d6, m, c); d7 = fma(d7, m, c);
      if (mixed) {
        a0 = (unsigned long long)(uint32_t)a0 * mi + a0; a1 = (unsigned long long)(uint32_t)a1 * mi + a1;
        a2 = (unsigned long long)(uint32_t)a2 * mi + a2; a3 = (unsigned long long)(uint32_t)a3 * mi + a3;
        a4 = (unsigned long long)(uint32_t)a4 * mi + a4; a5 = (unsigned long long)(uint32_t)a5 * mi + a5;
        a6 = (unsigned long long)(uint32_t)a6 * mi + a6; a7 = (unsigned long long)(uint32_t)a7 * mi + a7;
      }
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = d0 + d1 + d2 + d3 + d4 + d5 + d6 + d7 + (double)(a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7);
}
__attribute__((visibility("default"))) int bz_dfma_peak(bz_ctx* ctx, int mixed_with_imad_wide, double* ops_per_sec) {
  BZ_TRY(ctx, {
    BZ_CHECK(ops_per_sec, "null out");
    const int blocks = ctx->c.sm_count * 8, threads = 256;
    const uint32_t iters = 2048;
    bz::DevBuf out; out.alloc((size_t)blocks * threads * 8);
    cudaStream_t st = ctx->c.stream;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    dfma_peak_kernel<<<blocks, threads, 0, st>>>(out.as<double>(), 64, mixed_with_imad_wide);
    double best = 0;
    for (int rep = 0; rep < 3; ++rep) {
      cudaEventRecord(e0, st);
      dfma_peak_kernel<<<blocks, threads, 0, st>>>(out.as<double>(), iters, mixed_with_imad_wide);
      cudaEventRecord(e1, st);
      BZ_CUDA(cudaEventSynchronize(e1));
      float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
      double ops = (double)blocks * threads * iters * 64.0 * (mixed_with_imad_wide ? 2.0 : 1.0);
      best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    ctx->c.kernel_launches += 4;
    *ops_per_sec = best;
  });
}

__attribute__((visibility("default"))) int bz_imad_wide_peak(bz_ctx* ctx, double* imad_wide_per_sec) {
  BZ_TRY(ctx, {
    BZ_CHECK(imad_wide_per_sec, "null out");
    const int blocks = ctx->c.sm_count * 8, threads = 256;
    const uint32_t iters = 4096;
    bz::DevBuf out; out.alloc((size_t)blocks * threads * 8);
    cudaStream_t st = ctx->c.stream;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    imad_wide_peak_kernel<<<blocks, threads, 0, st>>>(out.as<unsigned long long>(), 64);
    double best = 0;
    for (int rep = 0; rep < 3; ++rep) {
      cudaEventRecord(e0, st);
      imad_wide_peak_kernel<<<blocks, threads, 0, st>>>(out.as<unsigned long long>(), iters);
      cudaEventRecord(e1, st);
      BZ_CUDA(cudaEventSynchronize(e1));
      float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
      double ops = (double)blocks * threads * iters * 64.0;
      best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    ctx->c.kernel_launches += 4;
    *imad_wide_per_sec = best;
  });
}

__attribute__((visibility("default"))) int bz_imad_peak(bz_ctx* ctx, double* imad_per_sec) {
  BZ_TRY(ctx, {
    BZ_CHECK(imad_per_sec, "null out");
    const int blocks = ctx->c.sm_count * 8, threads = 256;
    const uint32_t iters = 4096;
    bz::DevBuf out; out.alloc((size_t)blocks * threads * 4);
    cudaStream_t st = ctx->c.stream;
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    imad_peak_kernel<<<blocks, threads, 0, st>>>(out.as<uint32_t>(), 64);
    double best = 0;
    for (int rep = 0; rep < 3; ++rep) {
      cudaEventRecord(e0, st);
      imad_peak_kernel<<<blocks, threads, 0, st>>>(out.as<uint32_t>(), iters);
      cudaEventRecord(e1, st);
      BZ_CUDA(cudaEventSynchronize(e1));
      float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
      double ops = (double)blocks * threads * iters * 64.0;
      best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    ctx->c.kernel_launches += 4;
    *imad_per_sec = best;
  });
}

// ---- element-wise field / point ops on host slices ------------------------------------------------
__attribute__((visibility("default"))) int bz_field_op(bz_ctx* ctx, int field, int op, const void* a, const void* b, void* out, uint64_t n) {
  BZ_TRY(ctx, {
    BZ_CHECK(field == 0 || field == 1, "bad field id");
    BZ_CHECK(op >= 0 && op <= 9, "bad op");
    if (!n) return BZ_OK;
    BZ_CHECK(a && out, "null argument");
    BZ_CHECK(op > 2 || b, "binary field op without a second operand");
    BZ_CHECK(n <= (1ull << 32), "field op: slice too long");
    size_t in_sz = op == 4 ? 64 : 32;
    bz::DevBuf da, db, dout;
    da.alloc(n * in_sz + 32); db.alloc(n * 32 + 32); dout.alloc(n * 32 + 32);
    cudaStream_t st = ctx->c.stream;
    BZ_CUDA(cudaMemcpyAsync(da.p, a, n * in_sz, cudaMemcpyHostToDevice, st));
    if (b && op <= 2) BZ_CUDA(cudaMemcpyAsync(db.p, b, n * 32, cudaMemcpyHostToDevice, st));
    bz::field_op_run(&ctx->c, field, op, da.p, db.p, dout.p, n);
    BZ_CUDA(cudaMemcpyAsync(out, dout.p, n * 32, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}
__attribute__((visibility("default"))) int bz_batch_invert_assigned_dev(bz_ctx* ctx, int field, const void* d_num, const void* d_den, void* d_out, uint64_t n) {
  BZ_TRY(ctx, {
    BZ_CHECK(field == 0 || field == 1, "bad field id");
    bz::batch_invert_assigned_run(&ctx->c, field, d_num, d_den, d_out, n);
  });
}
__attribute__((visibility("default"))) int bz_batch_invert_assigned(bz_ctx* ctx, int field, const void* num, const void* den, void* out, uint64_t n) {
  BZ_TRY(ctx, {
    BZ_CHECK(field == 0 || field == 1, "bad field id");
    bz::DevBuf dn, dd;
    dn.alloc(n * 32 + 32); dd.alloc(n * 32 + 32);
    cudaStream_t st = ctx->c.stream;
    BZ_CUDA(cudaMemcpyAsync(dn.p, num, n * 32, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaMemcpyAsync(dd.p, den, n * 32, cudaMemcpyHostToDevice, st));
    bz::batch_invert_assigned_run(&ctx->c, field, dn.p, dd.p, dn.p, n);          // in place over the numerators
    BZ_CUDA(cudaMemcpyAsync(out, dn.p, n * 32, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}
__attribute__((visibility("default"))) int bz_curve_op(bz_ctx* ctx, int curve, int op, const void* a, const void* b, void* out, uint64_t n) {
  BZ_TRY(ctx, {
    BZ_CHECK(curve == 0 || curve == 1, "bad curve id");
    BZ_CHECK(op >= 0 && op <= 4, "bad op");
    bz::DevBuf da, db, dout;
    da.alloc(n * 64 + 64); db.alloc(n * 64 + 64); dout.alloc(n * 64 + 64);
    cudaStream_t st = ctx->c.stream;
    BZ_CUDA(cudaMemcpyAsync(da.p, a, n * 64, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaMemcpyAsync(db.p, b, n * 64, cudaMemcpyHostToDevice, st));
    bz::curve_op_run(&ctx->c, curve, op, da.p, db.p, dout.p, n);
    BZ_CUDA(cudaMemcpyAsync(out, dout.p, n * 64, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}

// ---- ChaCha20 keystream (the stream bz_create_proofs_seeded expands) --------------------------------
__attribute__((visibility("default"))) int bz_chacha20_blocks(bz_ctx* ctx, const void* seeds, uint32_t batch, uint64_t blocks_per_seed, void* out) {
  BZ_TRY(ctx, {
    BZ_CHECK(seeds && out, "null argument");
    if (!batch || !blocks_per_seed) return BZ_OK;
    BZ_CHECK(blocks_per_seed <= (SIZE_MAX / 64) / batch, "chacha20: output size overflows");
    const size_t bytes = (size_t)batch * blocks_per_seed * 64;
    cudaStream_t st = ctx->c.stream;
    bz::DevBuf &ds = ctx->c.stage[0], &dout = ctx->c.stage[1];
    ds.ensure((size_t)batch * 32);
    BZ_CUDA(cudaMemcpyAsync(ds.p, seeds, (size_t)batch * 32, cudaMemcpyHostToDevice, st));
    cudaPointerAttributes at{};
    const bool on_device = cudaPointerGetAttributes(&at, out) == cudaSuccess && at.type == cudaMemoryTypeDevice;
    cudaGetLastError();
    if (on_device && ((uintptr_t)out & 15) == 0) {
      bz::chacha20_fill_run(&ctx->c, ds.p, batch, blocks_per_seed, out);
    } else {
      dout.ensure(bytes);
      bz::chacha20_fill_run(&ctx->c, ds.p, batch, blocks_per_seed, dout.p);
      BZ_CUDA(cudaMemcpyAsync(out, dout.p, bytes, cudaMemcpyDefault, st));
    }
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}

// ---- MSM ----------------------------------------------------------------------------------------
__attribute__((visibility("default"))) int bz_msm_dev(bz_ctx* ctx, int curve, const void* d_coeffs, const void* d_bases, uint64_t n, void* d_out_jac, int window_bits) {
  BZ_TRY(ctx, {
    BZ_CHECK(curve == 0 || curve == 1, "bad curve id");
    BZ_CHECK(n < (1ull << 31), "msm: n too large");
    BZ_CHECK(window_bits == 0 || (window_bits >= 2 && window_bits <= 16), "msm: window_bits out of range");
    bz::msm_run(&ctx->c, curve, d_coeffs, d_bases, (uint32_t)n, d_out_jac, window_bits);
  });
}

__attribute__((visibility("default"))) int bz_best_multiexp(bz_ctx* ctx, int curve, const void* coeffs, const void* bases, uint64_t n, void* out_jac) {
  BZ_TRY(ctx, {
    BZ_CHECK(curve == 0 || curve == 1, "bad curve id");
    BZ_CHECK(n < (1ull << 31), "msm: n too large");
    bz::DevBuf &ds = ctx->c.stage[0], &db = ctx->c.stage[1], &dout = ctx->c.stage[2];
    ds.ensure(n * 32 + 32); db.ensure(n * 64 + 64); dout.ensure(96);
    cudaStream_t st = ctx->c.stream;
    BZ_CUDA(cudaMemcpyAsync(ds.p, coeffs, n * 32, cudaMemcpyHostToDevice, st));
    BZ_CUDA(cudaMemcpyAsync(db.p, bases, n * 64, cudaMemcpyHostToDevice, st));
    bz::msm_run(&ctx->c, curve, ds.p, db.p, (uint32_t)n, dout.p, 0);
    BZ_CUDA(cudaMemcpyAsync(out_jac, dout.p, 96, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}

__attribute__((visibility("default"))) int bz_point_sum_dev(bz_ctx* ctx, int curve, const void* d_jac, uint32_t count, void* d_out_affine) {
  BZ_TRY(ctx, {
    BZ_CHECK(curve == 0 || curve == 1, "bad curve id");
    BZ_CHECK(d_jac && d_out_affine && count >= 1 && count <= 4096, "point sum: bad arguments");
    bz::jac_sum_run(&ctx->c, curve, d_jac, count, d_out_affine);
  });
}

__attribute__((visibility("default"))) int bz_batch_normalize_dev(bz_ctx* ctx, int curve, const void* d_jac, void* d_affine, uint64_t n) {
  BZ_TRY(ctx, {
    BZ_CHECK(curve == 0 || curve == 1, "bad curve id");
    BZ_CHECK(n < (1ull << 32), "batch_normalize: too many points");
    BZ_CHECK(n == 0 || (d_jac && d_affine), "null argument");
    bz::jac_to_affine_run(&ctx->c, curve, d_jac, d_affine, (uint32_t)n);
  });
}

// ---- NTT ----------------------------------------------------------------------------------------
__attribute__((visibility("default"))) int bz_ntt_dev(bz_ctx* ctx, int field, const void* d_in, void* d_out, uint32_t log_n, int inverse, int batch) {
  BZ_TRY(ctx, {
    BZ_CHECK(field == 0 || field == 1, "bad field id");
    bz::NttFusion fu;
    bz::ntt_run(&ctx->c, field, d_in, d_out, (int)log_n, inverse != 0, batch, fu);
  });
}
__attribute__((visibility("default"))) int bz_lagrange_to_coeff_dev(bz_ctx* ctx, int field, const void* d_in, void* d_out, uint32_t k, int batch) {
  BZ_TRY(ctx, {
    BZ_CHECK(field == 0 || field == 1, "bad field id");
    bz::NttFusion fu; fu.post_mode = 1;
    bz::ntt_run(&ctx->c, field, d_in, d_out, (int)k, true, batch, fu);
  });
}
__attribute__((visibility("default"))) int bz_coeff_to_extended_dev(bz_ctx* ctx, int field, const void* d_in, void* d_out, uint32_t k, uint32_t extended_k, int batch) {
  BZ_TRY(ctx, {
    BZ_CHECK(field == 0 || field == 1, "bad field id");
    BZ_CHECK(extended_k >= k, "extended_k < k");
    bz::NttFusion fu; fu.n_in = extended_k > k ? (1ull << k) : 0; fu.pre_zeta = true;
    bz::ntt_run(&ctx->c, field, d_in, d_out, (int)extended_k, false, batch, fu);
  });
}
__attribute__((visibility("default"))) int bz_extended_to_coeff_dev(bz_ctx* ctx, int field, const void* d_in, void* d_out, uint32_t extended_k, int batch) {
  BZ_TRY(ctx, {
    BZ_CHECK(field == 0 || field == 1, "bad field id");
    bz::NttFusion fu; fu.post_mode = 3;
    bz::ntt_run(&ctx->c, field, d_in, d_out, (int)extended_k, true, batch, fu);
  });
}

static int host_ntt(bz_ctx* ctx, int field, const void* in, size_t n_in, void* out, size_t n_out, int logN, bool inverse, const bz::NttFusion& fu) {
  BZ_TRY(ctx, {
    BZ_CHECK(field == 0 || field == 1, "bad field id");
    bz::DevBuf &din = ctx->c.stage[0], &dout = ctx->c.stage[1];
    din.ensure(n_in * 32); dout.ensure(n_out * 32);
    cudaStream_t st = ctx->c.stream;
    BZ_CUDA(cudaMemcpyAsync(din.p, in, n_in * 32, cudaMemcpyHostToDevice, st));
    bz::ntt_run(&ctx->c, field, din.p, dout.p, logN, inverse, 1, fu);
    BZ_CUDA(cudaMemcpyAsync(out, dout.p, n_out * 32, cudaMemcpyDeviceToHost, st));
    BZ_CUDA(cudaStreamSynchronize(st));
  });
}

__attribute__((visibility("default"))) int bz_best_fft(bz_ctx* ctx, int field, void* a, const void* omega, uint32_t log_n) {
  if (!ctx) return BZ_ERR_INVALID;
  if ((field != 0 && field != 1) || log_n > 30) { ctx->c.last_error = "bad field id or log_n"; return BZ_ERR_INVALID; }
  const bzh::Field& F = ctx->c.field(field);
  bzh::Fe w = F.root_of_unity();
  for (uint32_t i = log_n; i < 32; ++i) w = F.sqr(w);
  bzh::Fe om; memcpy(om.l, omega, 32);
  bool inverse;
  if (om == w) inverse = false;
  else if (om == F.inv(w)) inverse = true;
  else { ctx->c.last_error = "bz_best_fft: omega is not the 2^log_n domain generator or its inverse"; return BZ_ERR_UNSUPPORTED; }
  bz::NttFusion fu;
  size_t n = (size_t)1 << log_n;
  return host_ntt(ctx, field, a, n, a, n, (int)log_n, inverse, fu);
}
__attribute__((visibility("default"))) int bz_lagrange_to_coeff(bz_ctx* ctx, int field, void* a, uint32_t k) {
  if (!ctx) return BZ_ERR_INVALID;
  bz::NttFusion fu; fu.post_mode = 1;
  size_t n = (size_t)1 << k;
  return host_ntt(ctx, field, a, n, a, n, (int)k, true, fu);
}
__attribute__((visibility("default"))) int bz_coeff_to_extended(bz_ctx* ctx, int field, const void* coeffs, void* out_extended, uint32_t k, uint32_t extended_k) {
  if (!ctx) return BZ_ERR_INVALID;
  if (extended_k < k) { ctx->c.last_error = "extended_k < k"; return BZ_ERR_INVALID; }
  bz::NttFusion fu; fu.n_in = extended_k > k ? (1ull << k) : 0; fu.pre_zeta = true;
  return host_ntt(ctx, field, coeffs, (size_t)1 << k, out_extended, (size_t)1 << extended_k, (int)extended_k, false, fu);
}
__attribute__((visibility("default"))) int bz_extended_to_coeff(bz_ctx* ctx, int field, void* a, uint32_t extended_k) {
  if (!ctx) return BZ_ERR_INVALID;
  bz::NttFusion fu; fu.post_mode = 3;
  size_t n = (size_t)1 << extended_k;
  return host_ntt(ctx, field, a, n, a, n, (int)extended_k, true, fu);
}

}  // extern "C"
