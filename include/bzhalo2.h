/* libbzhalo2 -- C ABI of the B200-native Halo2 (IPA / Pasta) prover hot path.
 *
 * This is the drop-in boundary for the path BASELINE.json names: the arithmetic that
 * `halo2_proofs 0.2.0` (pinned at /root/reference/Cargo.lock:382-393, not vendored) executes inside
 * `create_proof`, as called by the reference at
 *   /root/reference/benches/shot.rs:58-71, /root/reference/benches/board.rs:51-86,
 *   /root/reference/src/circuits/shot.rs:915-940, /root/reference/src/circuits/board.rs:907-932.
 * A patched halo2_proofs (INTEGRATION.md) binds these symbols one-for-one from
 * `arithmetic.rs`, `poly/domain.rs`, `poly/commitment.rs` and the prover modules.
 *
 * Data layout across the ABI (SURVEY §8b):
 *   field element : 32 B = pasta's in-memory [u64;4], little-endian, Montgomery form (R = 2^256)
 *                   -> `&[Fp]` / `&[Fq]` pass through with zero conversion
 *   affine point  : 64 B  x || y (Montgomery); identity = 64 zero bytes
 *   Jacobian point: 96 B  x || y || z (Montgomery); identity has z = 0
 *   field id      : 0 = Fp (pallas::Base = vesta::Scalar), 1 = Fq (pallas::Scalar = vesta::Base)
 *   curve id      : 0 = Vesta (scalars Fp, coordinates Fq) -- the commitment curve of Board/Shot
 *                   1 = Pallas (scalars Fq, coordinates Fp)
 * Every function returns 0 on success, <0 on failure (bz_last_error gives the message); no C++
 * exception or abort crosses the boundary.  A context is bound to one GPU and one CUDA stream and
 * may be used by one thread at a time; contexts are independent.  There is NO CPU fallback:
 * without a CUDA device bz_ctx_create fails.
 */
#ifndef BZHALO2_H
#define BZHALO2_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bz_ctx bz_ctx;

#define BZ_OK 0
#define BZ_ERR_INVALID (-1)
#define BZ_ERR_CUDA (-2)
#define BZ_ERR_UNSUPPORTED (-3)
#define BZ_ERR_SYNTHESIS (-4) /* maps to plonk::Error::ConstraintSystemFailure / Synthesis */

#define BZ_FIELD_FP 0
#define BZ_FIELD_FQ 1
#define BZ_CURVE_VESTA 0
#define BZ_CURVE_PALLAS 1

/* ---- context ---------------------------------------------------------------------------------- */
/* stream = a cudaStream_t owned by the caller (e.g. torch's current stream) or NULL for a private one */
int bz_ctx_create(int device, void* stream, bz_ctx** out);
void bz_ctx_destroy(bz_ctx* ctx);
const char* bz_last_error(bz_ctx* ctx);
int bz_sync(bz_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t bz_kernel_launches(bz_ctx* ctx);
const char* bz_version(void);

/* ---- one large proof across the GPUs of a box (SURVEY 8e: "independent column commitments ... sharded per GPU", "a large MSM
 * split by point range with one final NCCL point-sum") -----------------------------------------------------------------------
 * Every rank calls bz_create_proofs with IDENTICAL inputs.  The MSMs of each commitment batch (table path and bucket path alike)
 * are dealt out by column when the batch has at least `world` of them, otherwise each bucket MSM is split by point range; a rank
 * writes its partial sums (128-byte XYZZ / 96-byte Jacobian) into d_send (device memory, capacity_per_rank bytes) and calls
 * exchange(user, bytes), which must all-gather `bytes` bytes from every rank's d_send into d_recv (rank-major, world x bytes) ON
 * THE CONTEXT'S STREAM (e.g. ncclAllGather / torch.distributed.all_gather_into_tensor) and return 0.  For a batch of one proof,
 * h(X) on the extended coset is evaluated by point range as well when capacity_per_rank >= 14 * 2^k * 32 / world bytes (the
 * slices of the 8n / 4n / 2n evaluation tiers); with a smaller buffer it is computed redundantly.  Everything else of the
 * proof (NTTs, scans, transcript) is computed redundantly, so all ranks write the same proof bytes.  world = 1 switches it off. */
typedef int (*bz_allgather_fn)(void* user, size_t bytes_per_rank);
int bz_ctx_set_sharding(bz_ctx* ctx, uint32_t rank, uint32_t world, void* d_send, void* d_recv, size_t capacity_per_rank,
                        bz_allgather_fn exchange, void* user);

/* ---- per-kernel-class device timing (CUDA events on the context's stream) ------------------------ */
/* tags: 0 ntt_pass, 1 msm_digits, 2 msm_sort, 3 msm_bucket, 4 msm_reduce, 5 msm_combine, 6 fixed_msm,
 *       7 quotient, 8 scan, 9 eval, 10 poly, 11 ipa, 12 other */
int bz_profile_enable(bz_ctx* ctx, int on);
int bz_profile_read(bz_ctx* ctx, int tag, double* total_ms, uint64_t* count);
/* counters collected while profiling: 0 = mixed point additions executed by the fixed-base MSM kernel */
int bz_profile_counter(bz_ctx* ctx, int which, uint64_t* value, int reset);
/* measured integer multiply-add peak of this GPU (IMAD/s), the roofline denominator of the integer-bound kernels */
int bz_imad_peak(bz_ctx* ctx, double* imad_per_sec);
/* same for the 32x32+64->64 form (IMAD.WIDE.U32), which is what the field multiplication is built from */
int bz_imad_wide_peak(bz_ctx* ctx, double* imad_wide_per_sec);

/* FP64-pipe probe: DFMA/s alone (mixed = 0) or DFMA + IMAD.WIDE per second issued from the same warps (mixed = 1) */
int bz_dfma_peak(bz_ctx* ctx, int mixed_with_imad_wide, double* ops_per_sec);

/* ---- device memory (library-owned, freed by bz_dev_free or with the context) ------------------- */
int bz_dev_alloc(bz_ctx* ctx, size_t bytes, void** dptr);
int bz_dev_free(bz_ctx* ctx, void* dptr);
int bz_h2d(bz_ctx* ctx, void* dptr, const void* host, size_t bytes);
int bz_d2h(bz_ctx* ctx, void* host, const void* dptr, size_t bytes);

/* ---- ff::Field / group ops on host slices (pasta_curves semantics; used by the parity suite and by the
 * shim for the few scalar-sized steps it does not want to do on the CPU) ------------------------------ */
/* op: 0 a*b, 1 a+b, 2 a-b, 3 a^-1 over the slice (ff::BatchInvert: Montgomery trick, 0 -> 0), 4 from_u512 (a = n x 64 B little-endian), 5 Montgomery -> canonical,
 *     6 canonical -> Montgomery, 7 -a, 8 a^2, 9 a^-1 element-wise by binary GCD (gcdinv.h; same values as op 3) */
int bz_field_op(bz_ctx* ctx, int field, int op, const void* a, const void* b, void* out, uint64_t n);
/* poly::batch_invert_assigned (U: halo2_proofs 0.2.0 src/poly.rs `batch_invert_assigned`, called by create_proof on the
 * advice columns a circuit assigned as Assigned<F>; reference call path R:src/circuits/shot.rs:921 -> create_proof):
 * out[i] = num[i] / den[i] with ff::BatchInvert semantics (den = 0 -> 0).  Assigned::Zero is (0, 1), Trivial(x) is (x, 1).
 * Host slices; the _dev form takes device pointers (may alias out = num) and is asynchronous on the context's stream,
 * so the shim can write a whole advice region (num_advice x n) in one call straight where bz_create_proofs reads it. */
int bz_batch_invert_assigned(bz_ctx* ctx, int field, const void* numerators, const void* denominators, void* out, uint64_t n);
int bz_batch_invert_assigned_dev(bz_ctx* ctx, int field, const void* d_numerators, const void* d_denominators, void* d_out, uint64_t n);
/* affine in, affine out (64 B each): op 0 a+b, 1 2a, 2 a-b, 3 2a+b (full projective add), 4 [k]a, k = first u32 of b */
int bz_curve_op(bz_ctx* ctx, int curve, int op, const void* a, const void* b, void* out, uint64_t n);

/* ---- ChaCha20 keystream: the blinding randomness of bz_create_proofs_seeded ---------------------------------------------------
 * out[b][j] = ChaCha20 block j (64 B) of key seeds[b], for b < batch and j < blocks_per_seed: 20 rounds, key = the 32-byte seed,
 * a 64-bit block counter j in state words 12-13 and stream id 0 in words 14-15 (the original layout that rand_chacha's
 * ChaCha20Rng uses; for j < 2^32 it equals RFC 8439 with an all-zero nonce).  Block j is the 64-byte Scalar::random draw j
 * (8 x next_u64, low word first), so out has rand_wide's layout: batch x blocks_per_seed x 64 B.
 *   seeds : batch x 32 B (host).  A seed must come from a CSPRNG and never be reused.
 *   out   : host or device memory; 16-byte aligned device memory is written in place, without a copy.  Synchronous. */
int bz_chacha20_blocks(bz_ctx* ctx, const void* seeds, uint32_t batch, uint64_t blocks_per_seed, void* out);

/* ---- arithmetic::best_multiexp(coeffs, bases) -> C::Curve  (U: halo2_proofs/src/arithmetic.rs) -- */
/* host buffers; copies are part of the call.  out_jac: 96 B. */
int bz_best_multiexp(bz_ctx* ctx, int curve, const void* coeffs, const void* bases, uint64_t n, void* out_jac);
/* device-resident variant (all pointers from bz_dev_alloc); window_bits = 0 picks automatically */
int bz_msm_dev(bz_ctx* ctx, int curve, const void* d_coeffs, const void* d_bases, uint64_t n, void* d_out_jac,
               int window_bits);
/* Sum of `count` Jacobian points -> one affine point, all device pointers: the local half of the one real multi-GPU
 * exchange on this path -- a large MSM split by point range leaves one 96 B partial per rank; NCCL all-gathers them
 * (it has no elliptic-curve reduction) and every rank adds them here. */
int bz_point_sum_dev(bz_ctx* ctx, int curve, const void* d_jac, uint32_t count, void* d_out_affine);
/* group::Curve::batch_normalize: n Jacobian -> n affine (device pointers) */
int bz_batch_normalize_dev(bz_ctx* ctx, int curve, const void* d_jac, void* d_affine, uint64_t n);

/* ---- arithmetic::best_fft(a, omega, log_n)  (U: halo2_proofs/src/arithmetic.rs) ----------------- */
/* In-place, natural order in/out.  omega must be the domain generator ROOT_OF_UNITY^(2^(32-log_n))
 * or its inverse -- the only values halo2_proofs ever passes (EvaluationDomain::new, Params::new);
 * anything else returns BZ_ERR_UNSUPPORTED. */
int bz_best_fft(bz_ctx* ctx, int field, void* a, const void* omega, uint32_t log_n);
/* device-resident batched transform: `batch` arrays of 2^log_n elements, contiguous */
int bz_ntt_dev(bz_ctx* ctx, int field, const void* d_in, void* d_out, uint32_t log_n, int inverse, int batch);

/* ---- EvaluationDomain (U: halo2_proofs/src/poly/domain.rs) --------------------------------------- */
/* lagrange_to_coeff: inverse NTT of size 2^k with the 1/n scale fused into the last pass */
int bz_lagrange_to_coeff_dev(bz_ctx* ctx, int field, const void* d_in, void* d_out, uint32_t k, int batch);
/* coeff_to_extended: zeta^(i mod 3) pre-scale + zero-pad n -> 2^extended_k + forward NTT, one fused transform */
int bz_coeff_to_extended_dev(bz_ctx* ctx, int field, const void* d_in, void* d_out, uint32_t k, uint32_t extended_k,
                             int batch);
/* extended_to_coeff: inverse NTT of size 2^extended_k, 1/N and zeta^-(i mod 3) fused (caller truncates) */
int bz_extended_to_coeff_dev(bz_ctx* ctx, int field, const void* d_in, void* d_out, uint32_t extended_k, int batch);
/* host-buffer conveniences mirroring the Rust signatures (copies inside the call) */
int bz_lagrange_to_coeff(bz_ctx* ctx, int field, void* a, uint32_t k);
int bz_coeff_to_extended(bz_ctx* ctx, int field, const void* coeffs, void* out_extended, uint32_t k, uint32_t extended_k);
int bz_extended_to_coeff(bz_ctx* ctx, int field, void* a, uint32_t extended_k);

/* ==================================================================================================
 * The prover: Params / ProvingKey images on the device and `create_proof`
 * (U: halo2_proofs 0.2.0 src/poly/commitment.rs `Params`, src/plonk.rs `ProvingKey`, src/plonk/prover.rs
 *  `create_proof`; reference call sites /root/reference/benches/shot.rs:58-71).
 * ================================================================================================== */
typedef struct bz_params bz_params;
typedef struct bz_pk bz_pk;

/* Params<C>: g, g_lagrange (n affine points each), w, u -- exactly the fields of halo2's `Params` (host memory).
 * Builds the device image incl. the fixed-base window tables used by every commitment.
 * window_bits: signed-digit window of the tables (0 = default). */
int bz_params_create(bz_ctx* ctx, uint32_t k, int curve, const void* g, const void* g_lagrange, const void* w,
                     const void* u, int window_bits, bz_params** out);
void bz_params_destroy(bz_params* params);
/* Params::new(k) (U: halo2_proofs 0.2.0 src/poly/commitment.rs; reference call sites /root/reference/benches/shot.rs:58,
 * benches/board.rs:51, src/circuits/shot.rs:915, src/circuits/board.rs:907): g[i] = hash_to_curve("Halo2-Parameters")
 * (0x00 || i LE32), g_lagrange = group inverse FFT of g, w / u = hasher(0x01) / hasher(0x02) -- all computed on the
 * device.  Outputs (host): g, g_lagrange = 2^k x 64 B affine; w, u = 64 B. */
int bz_params_new(bz_ctx* ctx, uint32_t k, int curve, void* g, void* g_lagrange, void* w, void* u);
/* pasta_curves `C::hash_to_curve(domain_prefix)(message)` for `count` messages of msg_len bytes each (host); 64 B affine
 * out per message.  (U: pasta_curves 0.4.1 src/hashtocurve.rs; reference call site /root/reference/src/utils/pedersen.rs:20-22,
 * KATs /root/reference/src/utils/constants/fixed_bases/board_commit_v.rs:5-14.) */
int bz_hash_to_curve(bz_ctx* ctx, int curve, const char* domain_prefix, const void* messages, uint32_t msg_len,
                     uint64_t count, void* out_affine);
/* pasta_curves `GroupEncoding::to_bytes / from_bytes` for n points (host buffers): 32 B = x little-endian canonical,
 * bit 255 = parity of y, identity = 32 zero bytes -- the encoding of `Params::write / read` (k: u32 LE, then g,
 * g_lagrange, w, u compressed) and of the proof's points.  status[i]: 0 ok, 1 identity, 2 not a curve point. */
int bz_points_compress(bz_ctx* ctx, int curve, const void* affine, uint64_t n, void* out32);
int bz_points_decompress(bz_ctx* ctx, int curve, const void* in32, uint64_t n, void* out_affine, uint8_t* status);
/* Params::commit (lagrange_basis = 0) / Params::commit_lagrange (1): poly = n scalars (host), blind = 1 scalar;
 * result already normalised: 64 B affine (what `.to_affine()` / batch_normalize yields). */
int bz_params_commit(bz_ctx* ctx, bz_params* params, int lagrange_basis, const void* poly, const void* blind,
                     void* out_affine);

/* Batched, device-resident form: `count` polynomials (count x n scalars, contiguous) and `count` blinds in, `count` affine
 * points out -- all device pointers.  Independent column commitments are what a multi-GPU prover shards per GPU. */
int bz_params_commit_batch_dev(bz_ctx* ctx, bz_params* params, int lagrange_basis, const void* d_polys,
                               const void* d_blinds, uint32_t count, void* d_out_affine);

/* The constraint system `pk.vk.cs` flattened (SURVEY App. G).  Expressions are postfix token streams. */
typedef struct {
  uint32_t op; /* 0 Constant(a = constant index) 1 Advice(a = column, b = rotation) 2 Fixed 3 Instance 4 Negated 5 Sum
                  6 Product 7 Scaled(a = constant index) */
  uint32_t a;
  int32_t b;
} bz_token;

typedef struct {
  uint32_t k, num_advice, num_fixed, num_instance, degree, blinding_factors;
  uint32_t n_advice_queries;   const int32_t* advice_queries;   /* (column, rotation) pairs in registration order */
  uint32_t n_fixed_queries;    const int32_t* fixed_queries;
  uint32_t n_instance_queries; const int32_t* instance_queries;
  uint32_t n_perm_columns;     const uint32_t* perm_columns;    /* (kind, index) pairs; kind 0 advice 1 fixed 2 instance */
  uint32_t n_constants;        const void* constants;           /* 32 B Montgomery each */
  uint32_t n_tokens;           const bz_token* tokens;
  uint32_t n_gate_polys;       const uint32_t* gate_poly_offsets;  /* n_gate_polys + 1 offsets into tokens, gate order */
  uint32_t n_lookups;          const uint32_t* lookup_input_counts; const uint32_t* lookup_table_counts;
  const uint32_t* lookup_expr_offsets; /* offsets (total + 1) into tokens; per lookup: its inputs, then its tables */
  uint8_t vk_transcript_repr[32];      /* canonical LE scalar that vk.hash_into absorbs (opaque; SURVEY App. A step 0) */
} bz_circuit;

/* keygen_pk's device image: fixed_values = num_fixed x n scalars (Lagrange), sigma_values = n_perm_columns x n scalars
 * (pk.permutation.permutations), both host memory.  Polys, extended cosets, l0 / l_blind / l_last and the compiled
 * quotient program are derived on the device. */
int bz_pk_create(bz_ctx* ctx, bz_params* params, const bz_circuit* cs, const void* fixed_values,
                 const void* sigma_values, bz_pk** out);
/* Same, with the permutation argument assembled on the device (U: plonk/permutation/keygen.rs `Assembly::build_pk`):
 * mapping = n_perm_columns x n pairs (column', row') of u32 -- the copy-constraint cycles as `Assembly::copy` leaves
 * them; sigma_j[i] = delta^column' * omega^row' is computed by a kernel. */
int bz_pk_create_from_assembly(bz_ctx* ctx, bz_params* params, const bz_circuit* cs, const void* fixed_values,
                               const uint32_t* mapping, bz_pk** out);
/* keygen_vk's commitments (U: plonk/keygen.rs): commit_lagrange(column, Blind::default()) of every fixed column and
 * every permutation (sigma) column, normalised: num_fixed x 64 B and n_perm_columns x 64 B affine (host; either may be
 * NULL).  Computed once per pk with the fixed-base tables and cached. */
int bz_pk_vk_commitments(bz_ctx* ctx, bz_pk* pk, void* fixed_commitments, void* perm_commitments);
void bz_pk_destroy(bz_pk* pk);
uint32_t bz_pk_num_random(const bz_pk* pk); /* Scalar::random draws one create_proof makes (protocol order) */
uint32_t bz_pk_proof_size(const bz_pk* pk); /* bytes `transcript.finalize()` yields */
/* Static count of field multiplications one point of the compiled h(X) program costs in evaluation tier `tier`
 * (0: every point of the extended coset, 1: every second, 2: every fourth; the figure SURVEY 8d's quotient roofline is
 * computed from); 0 for an empty tier.  *points, if not NULL, receives the number of coset points of that tier. */
uint32_t bz_pk_quotient_muls(const bz_pk* pk, uint32_t tier, uint32_t* points);

/* h(X) as generated code.  The compiled program of evaluation tier `tier` for a constraint system -- host only, needs no GPU
 * and no context: scripts/gen_quotient_kernels.py calls it at build time and emits one straight-line sm_100a kernel per program
 * into csrc/gen_quotient.cu (registers instead of the interpreter's local-memory stack); a proving key whose program hashes to a
 * generated kernel uses it (bz_pk_quotient_generated = 1), every other circuit runs the interpreter.  code / rot may be NULL to
 * query the sizes. */
int bz_quotient_program(const bz_circuit* cs, uint32_t tier, uint32_t* code, uint32_t code_cap, uint32_t* n_code, int32_t* rot,
                        uint32_t rot_cap, uint32_t* n_rot, uint64_t* hash);
int bz_pk_quotient_generated(const bz_pk* pk, uint32_t tier);

/* create_proof for `batch` independent proofs of the same circuit, in lockstep on the device.
 *   instances : batch x num_instance x instance_stride scalars; instance_lens[num_instance] values are used
 *   advice    : batch x num_advice x n scalars (rows >= n - (blinding_factors + 1) are ignored: blinded)
 *   rand_wide : batch x bz_pk_num_random x 64 B -- the raw outputs `Scalar::random(&mut rng)` would consume, in
 *               the exact order create_proof draws them (the shim pre-draws: the count is shape-only)
 *   (instances / advice / rand_wide may be host pointers or device pointers from bz_dev_alloc)
 *   proofs    : batch x bz_pk_proof_size bytes (host), identical to what Blake2bWrite::finalize() returns
 * Errors: BZ_ERR_SYNTHESIS when a lookup input is missing from its table (Error::ConstraintSystemFailure). */
int bz_create_proofs(bz_ctx* ctx, bz_pk* pk, uint32_t batch, const void* instances, const uint32_t* instance_lens,
                     uint32_t instance_stride, const void* advice, const void* rand_wide, void* proofs);

/* bz_create_proofs with the blinding randomness drawn on the device: proof b has exactly the bytes bz_create_proofs gives for
 * rand_wide[b] = the ChaCha20 keystream of seeds[b] (bz_chacha20_blocks with blocks_per_seed = bz_pk_num_random), which is the
 * stream stock halo2 consumes from `rand_chacha::ChaCha20Rng::from_seed(seeds[b])`.  The caller uploads 32 bytes per proof
 * instead of bz_pk_num_random x 64.
 *   seeds     : batch x 32 B (host).  A seed must come from a CSPRNG and never be reused: the seed fixes every blind of the
 *               proof, so one seed for two witnesses breaks zero knowledge.
 *   instances, instance_lens, instance_stride, advice, proofs : as for bz_create_proofs
 * Errors: BZ_ERR_INVALID for a null argument, batch = 0 or two equal seeds in one call; otherwise as bz_create_proofs. */
int bz_create_proofs_seeded(bz_ctx* ctx, bz_pk* pk, uint32_t batch, const void* instances, const uint32_t* instance_lens,
                            uint32_t instance_stride, const void* advice, const void* seeds, void* proofs);

/* plonk::verify_proof (SingleVerifier semantics: one verdict per proof) for `batch` proofs of the same circuit
 * (U: halo2_proofs 0.2.0 src/plonk/verifier.rs and the argument verifiers; reference call sites
 * /root/reference/benches/board.rs:84, src/circuits/shot.rs:933-940, src/circuits/board.rs:925-932).
 *   instances : as for bz_create_proofs      proofs : batch x proof_len bytes (host)
 *   results   : batch bytes, 1 = Ok(()), 0 = Err(_) (malformed point / scalar, wrong length, failed opening)
 * Point decompression, the instance commitments, compute_s and the final multi-scalar check run on the device.
 * Through a proving key, keygen_vk's commitments are computed on the first call and cached; bz_verify_proofs_vk below
 * verifies from a verifying key alone. */
int bz_verify_proofs(bz_ctx* ctx, bz_pk* pk, uint32_t batch, const void* instances, const uint32_t* instance_lens,
                     uint32_t instance_stride, const void* proofs, uint32_t proof_len, uint8_t* results);

/* The verifying key (U: halo2_proofs 0.2.0 src/plonk.rs `VerifyingKey`): what a process that only verifies holds -- the
 * constraint system (its k, domain and vk.hash_into scalar in `cs`), keygen_vk's fixed commitments (num_fixed x 64 B) and
 * permutation commitments (n_perm_columns x 64 B), affine Montgomery as bz_pk_vk_commitments returns them (host memory; NULL
 * only for an empty list).  No fixed values, no sigma columns: creating a vk allocates no device memory, and verifying needs
 * no proving key.  `params` must outlive the vk.  BZ_ERR_INVALID for a null argument, cs.k != params' k, Pallas params, or a
 * commitment that has a coordinate >= q, is not on y^2 = x^3 + 5, or is the identity (keygen_vk's Blind::default() adds
 * [1]W, so a real vk never holds it). */
typedef struct bz_vk bz_vk;
int bz_vk_create(bz_ctx* ctx, bz_params* params, const bz_circuit* cs, const void* fixed_commitments,
                 const void* perm_commitments, bz_vk** out);
void bz_vk_destroy(bz_vk* vk);
uint32_t bz_vk_proof_size(const bz_vk* vk); /* bytes of one proof of this circuit */
/* bz_verify_proofs from a verifying key: same arguments, checks and verdicts */
int bz_verify_proofs_vk(bz_ctx* ctx, bz_vk* vk, uint32_t batch, const void* instances, const uint32_t* instance_lens,
                        uint32_t instance_stride, const void* proofs, uint32_t proof_len, uint8_t* results);

/* ==================================================================================================
 * Fine-grained prover arithmetic (SURVEY 8b "minimum export set"): one call per inner loop of halo2_proofs 0.2.0, what a
 * patched plonk/permutation/prover.rs, plonk/lookup/prover.rs, plonk/vanishing/prover.rs, poly/domain.rs,
 * poly/multiopen/prover.rs, poly/commitment/prover.rs and arithmetic.rs bind one-for-one when the whole-proof call
 * (bz_create_proofs) is not used.  All buffers are HOST memory in pasta's in-memory Montgomery form; the calls are
 * synchronous.  They run the same kernels as bz_create_proofs with a batch of one.
 * ================================================================================================== */
/* permutation::Argument::commit, the body for ONE column set (U: src/plonk/permutation/prover.rs): n = 2^k rows,
 * values[j] / sigmas[j] = the set's ncols (<= 8, i.e. cs degree <= 10) columns and their sigma columns (Lagrange values),
 * delta_omega0 = DELTA^(index of the set's first column), z0 = last_z of the previous set (ONE for the first).
 * out_z[0] = z0, out_z[i+1] = out_z[i] * prod_j (v_j[i] + delta_omega0 DELTA^j omega^i beta + gamma) / (v_j[i] + beta sigma_j[i] + gamma);
 * the division is halo2's batch_invert, which takes 1/0 as 0: a zero denominator at row i makes out_z[i+1..] zero;
 * the caller overwrites the last `blinding_factors` rows and reads last_z = z[n - blinding_factors - 1] like upstream. */
int bz_perm_product(bz_ctx* ctx, int field, uint32_t k, uint32_t ncols, const void* const* values, const void* const* sigmas,
                    const void* beta, const void* gamma, const void* delta_omega0, const void* z0, void* out_z);
/* lookup::Argument::commit_permuted -> permute_expression_pair (U: src/plonk/lookup/prover.rs): the theta-compressed input
 * and table expressions (n scalars each); rows [0, usable_rows) are permuted (A' sorted, S' aligned; App. A step 5), rows
 * above come back zero for the caller's blinding.  BZ_ERR_SYNTHESIS = an input value is missing from the table
 * (Error::ConstraintSystemFailure). */
int bz_lookup_permute(bz_ctx* ctx, int field, uint32_t k, uint32_t usable_rows, const void* compressed_input,
                      const void* compressed_table, void* out_permuted_input, void* out_permuted_table);
/* lookup::Permuted::commit_product: z[0] = 1, z[i+1] = z[i] (A[i] + beta)(S[i] + gamma) / ((A'[i] + beta)(S'[i] + gamma)); n scalars out;
 * 1/0 is taken as 0 as in bz_perm_product */
int bz_lookup_product(bz_ctx* ctx, int field, uint32_t k, const void* compressed_input, const void* compressed_table,
                      const void* permuted_input, const void* permuted_table, const void* beta, const void* gamma, void* out_z);
/* EvaluationDomain::divide_by_vanishing_poly (U: src/poly/domain.rs): a[i] *= t_evaluations[i mod 2^(extended_k - k)], in place,
 * a = 2^extended_k scalars in the extended Lagrange basis */
int bz_divide_by_vanishing(bz_ctx* ctx, int field, uint32_t k, uint32_t extended_k, void* a);
/* vanishing::Argument::construct up to the coefficients of h(X) (U: src/plonk/vanishing/prover.rs, the expression list of
 * src/plonk/prover.rs; App. A steps 11-12): polys = bz_pk_num_poly_slots(pk) x n coefficients in the order advice[0..G),
 * instance[0..I), per lookup (A', S', Z), permutation z per set; out_h = (degree - 1) * n coefficients (the pieces, in order) */
int bz_pk_quotient(bz_ctx* ctx, bz_pk* pk, const void* polys, const void* theta, const void* beta, const void* gamma,
                   const void* y, void* out_h);
uint32_t bz_pk_num_poly_slots(const bz_pk* pk);
/* arithmetic::eval_polynomial for `count` (polynomial, point) pairs in one launch: polys[i] = n coefficients, points = count scalars */
int bz_eval_many(bz_ctx* ctx, int field, uint64_t n, uint32_t count, const void* const* polys, const void* points, void* out);
/* arithmetic::kate_division(a, point): a = n coefficients, out_q = n - 1 coefficients of a(X) / (X - point), remainder dropped */
int bz_kate_div(bz_ctx* ctx, int field, uint64_t n, const void* a, const void* point, void* out_q);
/* acc = acc * x + poly over n coefficients (multiopen's q_set / q' / P accumulation, the fold of the h pieces) */
int bz_axpy(bz_ctx* ctx, int field, uint64_t n, void* acc, const void* x, const void* poly);
/* poly::commitment::create_proof, the folding loop (U: src/poly/commitment/prover.rs).  The caller (transcript side) keeps
 * S, xi, z and the blinds; the device keeps p', b and G' (as challenge products over the original generators).
 *   bz_ipa_begin : p_prime = n coefficients of P' = P + xi S with p'(x3) already subtracted from the constant term; b = powers of x3
 *   bz_ipa_round : L_j, R_j (affine, 64 B) for the current round, with the caller's blinds l_rand, r_rand and challenge z
 *   bz_ipa_fold  : the round's folds by u_j (and its inverse)
 *   bz_ipa_finish: c = p'[0] after the k-th fold; frees the state (bz_ipa_destroy frees it early) */
typedef struct bz_ipa bz_ipa;
int bz_ipa_begin(bz_ctx* ctx, bz_params* params, const void* p_prime, const void* x3, bz_ipa** out);
int bz_ipa_round(bz_ctx* ctx, bz_ipa* ipa, const void* z, const void* l_rand, const void* r_rand, void* out_l_affine,
                 void* out_r_affine);
int bz_ipa_fold(bz_ctx* ctx, bz_ipa* ipa, const void* u, const void* u_inv);
int bz_ipa_finish(bz_ctx* ctx, bz_ipa* ipa, void* out_c);
void bz_ipa_destroy(bz_ipa* ipa);

#ifdef __cplusplus
}
#endif
#endif /* BZHALO2_H */
