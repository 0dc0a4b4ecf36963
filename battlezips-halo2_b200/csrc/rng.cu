// ChaCha20 keystream expansion on the device: create_proof's blinding randomness from one 32-byte seed per proof
// (bz_create_proofs_seeded, bz_chacha20_blocks).  The stream is the one `rand_chacha::ChaCha20Rng::from_seed(seed)` yields
// (D. J. Bernstein's original layout): state = the four constants, the 8 key words = seed, a 64-bit block counter in words
// 12-13 starting at 0, and stream id 0 in words 14-15; for counters below 2^32 this is RFC 8439 with an all-zero nonce.
// One 64-byte block is one `Scalar::random` draw (8 x next_u64, low word first), so block j of seed b lands exactly where
// rand_wide[b][j] sits: the output is laid out like bz_create_proofs' rand_wide (batch x blocks x 64 B).
#include "common.h"

namespace bz {

__device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return __funnelshift_l(x, x, r); }

__device__ __forceinline__ void chacha_quarter(uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d) {
  a += b; d ^= a; d = rotl32(d, 16);
  c += d; b ^= c; b = rotl32(b, 12);
  a += b; d ^= a; d = rotl32(d, 8);
  c += d; b ^= c; b = rotl32(b, 7);
}

// One thread per 64-byte block: thread i computes block j = i mod blocks of seed b = i / blocks.  ALU only; the seed is two
// 16-byte loads and the block four 16-byte stores.
__global__ void chacha20_blocks_kernel(const uint4* __restrict__ seeds, uint64_t blocks, uint64_t total, uint4* __restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const uint64_t b = i / blocks, j = i - b * blocks;
  const uint4 k0 = seeds[2 * b], k1 = seeds[2 * b + 1];
  const uint32_t s[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u,       // "expand 32-byte k"
                          k0.x, k0.y, k0.z, k0.w, k1.x, k1.y, k1.z, k1.w,
                          (uint32_t)j, (uint32_t)(j >> 32), 0u, 0u};
  uint32_t x[16];
#pragma unroll
  for (int w = 0; w < 16; ++w) x[w] = s[w];
#pragma unroll 1
  for (int r = 0; r < 10; ++r) {
    chacha_quarter(x[0], x[4], x[8], x[12]);
    chacha_quarter(x[1], x[5], x[9], x[13]);
    chacha_quarter(x[2], x[6], x[10], x[14]);
    chacha_quarter(x[3], x[7], x[11], x[15]);
    chacha_quarter(x[0], x[5], x[10], x[15]);
    chacha_quarter(x[1], x[6], x[11], x[12]);
    chacha_quarter(x[2], x[7], x[8], x[13]);
    chacha_quarter(x[3], x[4], x[9], x[14]);
  }
  uint4* o = out + i * 4;
#pragma unroll
  for (int q = 0; q < 4; ++q)
    o[q] = make_uint4(x[4 * q] + s[4 * q], x[4 * q + 1] + s[4 * q + 1], x[4 * q + 2] + s[4 * q + 2], x[4 * q + 3] + s[4 * q + 3]);
}

// d_seeds: B x 32 B, d_out: B x blocks x 64 B, both device memory and 16-byte aligned; asynchronous on the context's stream.
void chacha20_fill_run(Ctx* ctx, const void* d_seeds, uint32_t B, uint64_t blocks, void* d_out) {
  const uint64_t total = (uint64_t)B * blocks;
  if (!total) return;
  BZ_CHECK(((uintptr_t)d_seeds & 15) == 0 && ((uintptr_t)d_out & 15) == 0, "chacha20: buffers must be 16-byte aligned");
  const unsigned threads = 256;
  const uint64_t grid = (total + threads - 1) / threads;
  BZ_CHECK(grid < (1ull << 31), "chacha20: too many blocks for one launch");
  ProfScope ps(ctx, PROF_OTHER);
  chacha20_blocks_kernel<<<(unsigned)grid, threads, 0, ctx->stream>>>((const uint4*)d_seeds, blocks, total, (uint4*)d_out);
  ctx->kernel_launches++;
  BZ_CUDA(cudaGetLastError());
}

}  // namespace bz
