// Shared internal declarations of libbzhalo2 (not part of the C ABI; see include/bzhalo2.h).
#pragma once
#include <cuda_runtime.h>
#include <chrono>
#include <cstdio>
#include <cstdint>
#include <cstdio>
#include <map>
#include <memory>
#include <set>
#include <mutex>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>
#include "host_field.h"
#include <nvtx3/nvToolsExt.h>

namespace bz {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define BZ_CUDA(expr)                                                                                   \
  do {                                                                                                  \
    cudaError_t _e = (expr);                                                                            \
    if (_e != cudaSuccess)                                                                              \
      throw ::bz::Error(-2, std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                                std::to_string(__LINE__));                                              \
  } while (0)

#define BZ_CHECK(cond, msg)                                  \
  do {                                                       \
    if (!(cond)) throw ::bz::Error(-1, std::string(msg));    \
  } while (0)

// cudaFuncSetAttribute and occupancy queries act on the CURRENT device's copy of a kernel: a process that opens contexts on
// several GPUs (bz_ctx_create(device, ...)) must repeat them per device.  One instance per call site; `fn` runs once per device.
constexpr int BZ_MAX_DEVICES = 64;
struct PerDeviceOnce {
  std::mutex m;
  uint64_t done = 0;
  template <class F> void run(int device, F&& fn) {
    std::lock_guard<std::mutex> g(m);
    if (device < 0 || device >= BZ_MAX_DEVICES) { fn(); return; }
    if (!((done >> device) & 1)) { fn(); done |= 1ull << device; }
  }
};

// device buffer owned by a context (freed with it)
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept { release(); p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0; return *this; }
  ~DevBuf() { release(); }
  void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
  void alloc(size_t n) { release(); if (n) { BZ_CUDA(cudaMalloc(&p, n)); bytes = n; } }
  void ensure(size_t n) { if (n > bytes) alloc(n); }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct NttTableKey {
  int field, inverse, logM;
  bool operator<(const NttTableKey& o) const { return std::tie(field, inverse, logM) < std::tie(o.field, o.inverse, o.logM); }
};
struct NttTable { DevBuf lo, hi; };

// Per-kernel-class device timing (CUDA events on the launching stream), switched on by bz_profile_enable:
// bench.py reads the dominant kernel's average launch duration from here for the roofline object.
enum ProfTag { PROF_NTT_PASS = 0, PROF_MSM_DIGITS, PROF_MSM_SORT, PROF_MSM_BUCKET, PROF_MSM_REDUCE, PROF_MSM_COMBINE,
               PROF_FIXED_MSM, PROF_QUOTIENT, PROF_SCAN, PROF_EVAL, PROF_POLY, PROF_IPA, PROF_OTHER, PROF_NTAGS };
struct ProfRec { cudaEvent_t a, b; int tag; };

// One context = one GPU + one stream.  Callable from one thread at a time (SURVEY §8b).
struct Ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  int sm_count = 148;
  std::string last_error;
  bzh::Field fp{0}, fq{1};

  // NTT tables: wsmall[field][inverse] = w_{4096}^{+-i}, i < 2048; inter-pass tables by (field, inverse, logM)
  DevBuf wsmall[2][2];
  std::map<NttTableKey, NttTable> ntt_tables;
  DevBuf ntt_tmp;          // ping-pong scratch for multi-pass transforms
  DevBuf scratch[4];       // general reusable scratch (msm, staging)
  DevBuf stage[6];         // device staging of the host-buffer entry points (kept across calls: no cudaMalloc/cudaFree per call)
  DevBuf commit_jac;       // Jacobian results of params_commit_run's bucket MSM
  uint64_t kernel_launches = 0;   // counted by every launch site (bench.py's gpu_launches)
  bool profiling = false;
  DevBuf counters;        // [0] = mixed additions done by fixed_msm_kernel while profiling
  std::vector<ProfRec> prof;
  double prof_ms[PROF_NTAGS] = {0};
  uint64_t prof_count[PROF_NTAGS] = {0};

  // One large proof across the GPUs of a box (bz_ctx_set_sharding, SURVEY 8e): every rank runs the same create_proof; the MSMs
  // of a commitment batch are dealt out by column, or split by point range when there are fewer MSMs than ranks, and the
  // 96-byte Jacobian results are exchanged by the caller's all-gather (NCCL) on this context's stream.
  uint32_t shard_rank = 0, shard_world = 1;
  void* shard_send = nullptr; void* shard_recv = nullptr; size_t shard_cap = 0;
  int (*shard_exchange)(void*, size_t) = nullptr; void* shard_user = nullptr;

  const bzh::Field& field(int f) const { return f == 0 ? fp : fq; }
  ~Ctx();
};

// NVTX range (header-only nvtx3; a no-op unless a profiler is attached): prover phases and kernel classes show up by name
// in Nsight timelines and can be used as ncu range filters
// BZ_PHASE_TIMES=1 (diagnosis only): every phase range also prints its wall time, device drained at both ends
inline bool phase_times_enabled() { static const bool on = [] { const char* e = getenv("BZ_PHASE_TIMES"); return e && atoi(e) != 0; }(); return on; }
struct NvtxRange {
  const char* name_;
  std::chrono::steady_clock::time_point t0_;
  explicit NvtxRange(const char* name) : name_(name) {
    nvtxRangePushA(name);
    if (phase_times_enabled()) { cudaDeviceSynchronize(); t0_ = std::chrono::steady_clock::now(); }
  }
  ~NvtxRange() {
    if (phase_times_enabled()) {
      cudaDeviceSynchronize();
      fprintf(stderr, "[phase] %-60s %9.3f ms\n", name_, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0_).count());
    }
    nvtxRangePop();
  }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};
inline const char* prof_tag_name(int tag) {
  static const char* names[] = {"ntt_pass", "msm_digits", "msm_sort", "msm_bucket", "msm_reduce", "msm_combine", "fixed_msm", "quotient",
                                "scan", "eval", "poly", "ipa", "other"};
  return tag >= 0 && tag < (int)(sizeof(names) / sizeof(names[0])) ? names[tag] : "?";
}

// RAII scope: records a start/stop event pair around the launches issued inside it (only when profiling)
struct ProfScope {
  Ctx* c; ProfRec r; bool on;
  ProfScope(Ctx* ctx, int tag) : c(ctx), on(ctx->profiling) {
    nvtxRangePushA(prof_tag_name(tag));
    if (!on) return;
    r.tag = tag;
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, c->stream);
  }
  ~ProfScope() {
    nvtxRangePop();
    if (!on) return;
    cudaEventRecord(r.b, c->stream);
    c->prof.push_back(r);
  }
};

constexpr int WSMALL_LOG = 12;

// ---- ntt.cu ----
struct NttFusion {
  // input side (first pass): zero padding + coset pre-scale by zeta^(i mod 3)
  uint64_t n_in = 0;        // 0: input has N elements; else input has n_in (< N, power of two) elements, rest zero
  bool pre_zeta = false;    // multiply input coefficient i by zeta^(i mod 3)  (coeff_to_extended)
  // output side (last pass)
  int post_mode = 0;        // 0 none, 1 scale by N^-1 (ifft), 3 scale by N^-1 * zeta^-(i mod 3) (extended_to_coeff)
};
// Transform `batch` polynomials.  in: batch x n_in(or N) elements, out: batch x N elements (may alias in when
// n_in == 0).  Natural order in, natural order out.  omega = primitive 2^logN-th root from the field's
// ROOT_OF_UNITY (inverse -> its inverse).
// Optional outer batch (e.g. proofs): batch2 groups at in_stride2 / out_stride2 ELEMENTS apart, each holding `batch`
// contiguous arrays.
void ntt_run(Ctx* ctx, int field, const void* in, void* out, int logN, bool inverse, int batch, const NttFusion& fu,
             int batch2 = 1, uint64_t in_stride2 = 0, uint64_t out_stride2 = 0);

}  // namespace bz

// the opaque handle of the C ABI
struct bz_ctx {
  bz::Ctx c;
  bool own_stream = false;
  std::set<void*> allocs;
};
