/* bpg.h -- C ABI of libbpg: the B200-native (sm_100a) hot path under the Bulletproofs R1CS prover and
 * verifier of MarcKloter/bulletproofs_gadgets.
 *
 * Each entry point names the reference interface it replaces (file:line under /root/reference; "ext" = the call
 * lands in the un-vendored crates curve25519-dalek 1.x / bulletproofs `develop` / merlin 1.x, Cargo.toml:8,10,17-20,
 * so the citation is the reference's call site).  INTEGRATION.md shows the Rust `extern "C"` block and the patch
 * points in the fork that bind these symbols.
 *
 * Conventions
 *   - scalars: 32-byte little endian.  Inputs follow dalek `Scalar::from_bits` semantics (conversions.rs:18,43):
 *     any value < 2^256 is accepted and reduced mod l on the device; outputs are canonical (< l).
 *   - points: 32-byte compressed ristretto255 (dalek CompressedRistretto) unless stated otherwise.
 *   - return value: BPG_OK (0) or a negative BPG_E_* code; nothing throws or aborts across the ABI.
 *   - a bpg_ctx is bound to one CUDA device and one stream, and is NOT thread-safe; distinct contexts are
 *     independent.  The caller owns every host buffer.  No randomness is generated inside the library:
 *     every random value the reference draws from thread_rng is an explicit input (ext_rng32 / blindings).
 *   - there is no CPU fallback: every entry point that computes fails with BPG_E_CUDA without a device.
 */
#ifndef BPG_H
#define BPG_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define BPG_OK 0
#define BPG_E_CUDA (-1)        /* CUDA runtime error (see bpg_last_error) */
#define BPG_E_SIZE (-2)        /* bad size / capacity (R1CSError::InvalidGeneratorsLength) */
#define BPG_E_DECOMPRESS (-3)  /* a point encoding failed to decompress */
#define BPG_E_ARG (-4)         /* null / inconsistent argument */
#define BPG_E_FORMAT (-5)      /* R1CSProof::from_bytes failure (R1CSError::FormatError) */
#define BPG_E_NOMEM (-6)
#define BPG_E_COMM (-7)        /* NCCL not available / communicator error */

typedef struct bpg_ctx bpg_ctx;
typedef struct bpg_circuit bpg_circuit;

/* flags for bpg_r1cs_prove / bpg_r1cs_verify */
#define BPG_FLAG_LEGACY_FRAMING 1u /* proof bytes without the 1-byte phase tag, 14 fixed fields (SURVEY App. A.5) */
#define BPG_FLAG_WITNESS_ON_DEVICE 4u /* aL, aR, aO are device pointers to reduced scalars (HBM-resident timing) */
#define BPG_FLAG_FAST_BLINDING 2u  /* s_L, s_R expanded on the device from a transcript-derived seed instead of
                                      2n sequential Merlin TranscriptRng draws: valid proofs, different bytes */
/* Inner-product argument: after the first rounds the folded generators G^(k), H^(k) (512 each) are materialised once by a
 * multi-output MSM and the remaining rounds run over them (same L_j, R_j bytes, ~1/3 fewer point additions per proof).
 * On by default for padded sizes >= 2^15; these two flags force it off / on (any size >= 4) for tests and A/B timing. */
#define BPG_FLAG_NO_LATE_FOLD 8u
#define BPG_FLAG_FORCE_LATE_FOLD 16u

int bpg_ctx_create(int device, bpg_ctx **out);
void bpg_ctx_destroy(bpg_ctx *ctx);
const char *bpg_last_error(bpg_ctx *ctx);
const char *bpg_strerror(int code);
/* kernels launched by this context so far (bench.py reports the delta as gpu_launches) */
uint64_t bpg_launch_count(bpg_ctx *ctx);
int bpg_sync(bpg_ctx *ctx);
/* How host threads wait for the device (process-wide; initial value from the environment, BPG_BLOCKING_SYNC=1):
 * 0 = spin (lowest latency for one caller), 1 = sleep on an event (many provers per GPU: leaves the cores to the transcript RNG) */
void bpg_set_blocking_sync(int on);
/* Kernel sizing of the protocol calls (process-wide): -1 = automatic (throughput sizing while >= 4 prove / verify calls are
 * in flight in this process, latency sizing otherwise), 0 = latency (two-wave accumulate grids, shallow bucket reductions),
 * 1 = throughput (half-wave grids of long chunks, work-lean reductions; for several processes sharing one GPU).
 * Results are identical in every mode. */
void bpg_set_sizing_mode(int mode);

/* BulletproofGens::new(capacity, 1) + PedersenGens::default()  [ext; prover.rs:53,92  verifier.rs:89].
 * Derives the G/H chains (SHAKE256 stream on the host, double-Elligator on the device) and builds the resident
 * window tables in HBM.  Idempotent; growing re-derives. */
int bpg_gens_ensure(bpg_ctx *ctx, size_t capacity);
size_t bpg_gens_capacity(bpg_ctx *ctx);
/* compressed generators G[i0..i0+n), H[i0..i0+n) (for parity tests / BulletproofGens accessors) */
int bpg_gens_export(bpg_ctx *ctx, size_t i0, size_t n, uint8_t *G32, uint8_t *H32);
int bpg_pedersen_gens(bpg_ctx *ctx, uint8_t B32[32], uint8_t Bblinding32[32]);

/* PedersenGens::commit(v, r) batched: out[i] = compress(v[i]*B + r[i]*B~)
 * [ext; gadget.rs:31  commitments.rs:27,39  cs_buffer.rs:39  assignment_parser.rs:162] */
int bpg_pedersen_commit(bpg_ctx *ctx, const uint8_t *v, const uint8_t *r, size_t n, uint8_t *out32);

/* RistrettoPoint::vartime_multiscalar_mul / optional_multiscalar_mul over arbitrary points [ext].
 * BPG_E_DECOMPRESS if any point fails to decode (optional_multiscalar_mul returning None). */
int bpg_msm(bpg_ctx *ctx, const uint8_t *scalars, const uint8_t *points32, size_t n, uint8_t out32[32]);
/* sum sG[i]*G[offset+i] + sum sH[i]*H[offset+i] + sum extra_scalars[j]*extra_points[j]  (sG or sH may be NULL):
 * the shape of every MSM inside Prover::prove / Verifier::verify [ext; prover.rs:93 verifier.rs:90]. */
int bpg_msm_gens(bpg_ctx *ctx, const uint8_t *sG, const uint8_t *sH, size_t n, size_t offset,
                 const uint8_t *extra_scalars, const uint8_t *extra_points32, size_t k, uint8_t out32[32]);
/* same, scalars already resident on the device (n x 32 B each, device pointers); used for HBM-resident timing */
int bpg_msm_gens_dev(bpg_ctx *ctx, const void *d_sG, const void *d_sH, size_t n, size_t offset, uint8_t out32[32]);
/* partial sum as an uncompressed extended point (128 B) for multi-GPU point-range splits, and the combiner */
int bpg_msm_gens_partial_dev(bpg_ctx *ctx, const void *d_sG, const void *d_sH, size_t n, size_t offset, uint8_t out128[128]);
int bpg_points_sum_compress(bpg_ctx *ctx, const uint8_t *ext128, size_t n, uint8_t out32[32]);
/* ONE proof split over the ranks of a node (BASELINE configs[3]: a 2^20-multiplier circuit on 1/2/4/8 GPUs).  Every rank calls
 * bpg_r1cs_prove with the SAME arguments; each evaluates only its point range of every large MSM (commitments, IPP rounds, the
 * late-fold materialisation), writes its partial points (128 B each) to d_send, calls allgather(user, bytes) -- which must gather
 * d_send[0, bytes) of all ranks into d_recv in rank order and be complete on return (NCCL all-gather on NVLink in this repo,
 * bulletproofs_gadgets_b200/parallel.py) -- and adds the world partials.  The sums are group elements, so every rank derives
 * the same challenges and returns the same proof bytes as an unsharded prover.  send_cap >= 256 KiB (2 MiB lets the late fold
 * keep N / 256 generators at N = 2^20), d_recv >= world * send_cap.
 * world = 1 switches it off. */
typedef int (*bpg_allgather_fn)(void *user, size_t bytes_per_rank);
int bpg_ctx_set_shard(bpg_ctx *ctx, int rank, int world, void *d_send, void *d_recv, size_t send_cap, bpg_allgather_fn allgather, void *user);

/* The same sharding with the exchange INSIDE the library (SURVEY 8b bpg_comm_init): the context owns an NCCL communicator and
 * enqueues ncclAllGather of the partial points on its own stream between the producing kernel and the summing kernel -- no host
 * synchronisation, no callback.  NCCL is resolved at run time (dlopen libnccl.so.2; BPG_NCCL_LIB overrides the name).
 * Rank 0 calls bpg_comm_unique_id and distributes the 128 bytes (any channel); then EVERY rank calls bpg_comm_init (collective).
 * Afterwards bpg_r1cs_prove on these contexts is one proof over `world` GPUs exactly as with bpg_ctx_set_shard, and
 * bpg_msm_gens_sharded_dev is one MSM split by point range: d_sG / d_sH point at this rank's slice (n_local terms starting at
 * generator `offset`), every rank returns the same 32 bytes. */
int bpg_comm_unique_id(uint8_t out128[128]);
int bpg_comm_init(bpg_ctx *ctx, int rank, int world, const uint8_t id128[128]);
int bpg_comm_destroy(bpg_ctx *ctx);
int bpg_msm_gens_sharded_dev(bpg_ctx *ctx, const void *d_sG, const void *d_sH, size_t n_local, size_t offset, uint8_t out32[32]);

/* the same two steps with the 128-byte partial points staying on the device, for callers whose collective runs there
 * (NCCL all-gather of the partials through torch.distributed): the partial is written to d_out128 (complete when the
 * call returns), and the sum reads n gathered partials from d_ext128 (the caller orders it after its collective) */
int bpg_msm_gens_partial_to_dev(bpg_ctx *ctx, const void *d_sG, const void *d_sH, size_t n, size_t offset, void *d_out128);
int bpg_points_sum_compress_dev(bpg_ctx *ctx, const void *d_ext128, size_t n, uint8_t out32[32]);

/* One inner-product-argument generator fold: out[i] = sl*PL[i] + sr*PR[i]  (InnerProductProof::create's
 * G'/H' update, dalek: a 2-point vartime MSM per element) [ext; inside prover.rs:93]. */
int bpg_fold_points(bpg_ctx *ctx, const uint8_t sl[32], const uint8_t sr[32], const uint8_t *PL32, const uint8_t *PR32,
                    size_t n, uint8_t *out32);

/* MiMC (src/mimc_hash/mimc.rs:7-97, mimc_consts.rs).  The 486 round constants are data of the reference crate:
 * the caller installs them once (32-byte LE each, Scalar::from_bits). */
int bpg_mimc_set_constants(bpg_ctx *ctx, const uint8_t *consts486x32);
/* mimc_hash(preimage) for n byte strings: data = concatenation, offsets[n+1] byte offsets  [mimc.rs:61-75;
 * callers prover.rs:171,197,325 verifier.rs:451] */
int bpg_mimc_hash_batch(bpg_ctx *ctx, const uint8_t *data, const uint64_t *offsets, size_t n, uint8_t *out32);
/* unpadded sponge over 32-byte LE blocks (Merkle nodes, merkle_tree_gadget.rs:7-12,106): hash i absorbs blocks
 * [block_off[i], block_off[i+1]).  trace (nullable) receives the in-circuit witness of every absorbed block:
 * 972 multipliers x (a_L, a_R, a_O) x 32 B in gadget order (mimc_hash_gadget.rs:133-144). */
int bpg_mimc_sponge_batch(bpg_ctx *ctx, const uint8_t *blocks, const uint32_t *block_off, size_t n, uint8_t *out32,
                          uint8_t *trace);

/* Constraint system in flat CSR form: constraint r is sum_k coeff[k]*var[k] = 0 for k in [row_ptr[r], row_ptr[r+1]),
 * term_var = kind << 29 | index with kind 0=a_L 1=a_R 2=a_O 3=V 4=One  (bulletproofs r1cs::Variable /
 * LinearCombination as recorded by ConstraintSystem::constrain; cs_buffer.rs:89-113).  The library keeps a
 * column-major copy on the device. */
int bpg_circuit_create(bpg_ctx *ctx, size_t n_multipliers, size_t m_commitments, size_t q_constraints,
                       const uint32_t *row_ptr, const uint32_t *term_var, const uint8_t *term_coeff, bpg_circuit **out);
void bpg_circuit_destroy(bpg_circuit *c);

/* Witness evaluation on the device (SURVEY 8 f-3).  Multiplier i created by ConstraintSystem::multiply(left_i, right_i) has
 * a_L[i] = <left_i>, a_R[i] = <right_i>, a_O[i] = a_L[i] a_R[i], the linear combinations being evaluated over the assignment so
 * far [cs_buffer.rs:94-97 -> ext Prover::multiply, replayed by prover.rs:102-117].  lc_ptr[2n + 1]: the terms of left_0, right_0,
 * left_1, ... inside term_var / term_coeff (encoding as for bpg_circuit_create); a term may reference committed values (v, m of
 * them), One, and multipliers with a SMALLER index only.  Multipliers made by allocate_multiplier / allocate have an empty pair
 * of combinations: their a_L, a_R are inputs (aL, aR are in/out, n x 32 bytes), a_O is computed.  The dependency graph is
 * levelised on the host; a wide level is one launch (independent multipliers in parallel), a run of narrow levels one
 * single-block launch. */
int bpg_witness_eval(bpg_ctx *ctx, size_t n, size_t m, const uint32_t *lc_ptr, const uint32_t *term_var, const uint8_t *term_coeff,
                     const uint8_t *v, uint8_t *aL, uint8_t *aR, uint8_t *aO);

/* Prover::new(label) + commit(v_i, blinding_i)* + (constraints) + prove(&bp_gens)  [ext; prover.rs:52-54,93
 * gadget.rs:18-38].  Writes the m commitments to V_out (nullable) and the serialised R1CSProof to `proof`;
 * returns the proof length (> 0) or a negative BPG_E_* code.  ext_rng32 are the 32 bytes the reference's
 * TranscriptRngBuilder::finalize draws from thread_rng. */
long bpg_r1cs_prove(bpg_ctx *ctx, bpg_circuit *c, const uint8_t *label, size_t label_len, const uint8_t *aL,
                    const uint8_t *aR, const uint8_t *aO, const uint8_t *v, const uint8_t *v_blinding,
                    const uint8_t ext_rng32[32], unsigned flags, uint8_t *V_out, uint8_t *proof, size_t proof_cap);
/* Pipelining hint for a prover that knows its NEXT proof (a queue of jobs).  The 2n transcript-RNG draws behind s_L, s_R are
 * sequential (one Keccak-f each, ~0.7 s of one host core at n = 2^20) and nothing of a proof can overlap its own draws; this call
 * starts them for a FUTURE proof in the background -- it commits the openings (one small kernel), then a host thread draws the
 * stream through the lane-batched RNG service and stages it in HBM on the context's second stream -- and returns at once, so
 * the draws of proof k+1 hide behind the device work of proof k on the same context.  The next bpg_r1cs_prove on this context
 * whose (circuit, label, v_blinding, ext_rng32) are the same picks the stream up; proof bytes are identical with or without
 * the hint.  Up to two proofs can be pending; further hints are ignored.  flags as for bpg_r1cs_prove. */
int bpg_r1cs_prove_prefetch(bpg_ctx *ctx, bpg_circuit *c, const uint8_t *label, size_t label_len, const uint8_t *v,
                            const uint8_t *v_blinding, const uint8_t ext_rng32[32], unsigned flags);
/* K independent proofs in one call.  Proof i is byte-identical to
 * bpg_r1cs_prove(ctx, circuits[i], labels[i], label_lens[i], aL[i], aR[i], aO[i], v[i], v_blinding[i],
 *                ext_rng32 + 32 i, flags, V_out[i], proofs[i], proof_caps[i])
 * and its length is written to proof_lens[i].  The proofs of padded size N <= 4096 run through the phases of Prover::prove in
 * lockstep: each phase is one set of launches and one host round trip for all of them (5 + max lg N round trips per pass,
 * independent of the count); a proof with a larger N is proved by bpg_r1cs_prove inside the call, so any mix may be passed.
 *  - Every argument of every proof is checked before any device work: a NULL array or entry where bpg_r1cs_prove needs a
 *    pointer (V_out and its entries may be NULL), proof_caps[i] below the size of proof i or a generator capacity below N_i
 *    fail the whole call with the code bpg_r1cs_prove returns (BPG_E_ARG / BPG_E_SIZE) for the first such proof; nothing is
 *    written then and proof_lens is zeroed.  count = 0 returns BPG_OK.
 *  - flags: 0, BPG_FLAG_LEGACY_FRAMING, BPG_FLAG_NO_LATE_FOLD (a no-op at the batched sizes).  BPG_FLAG_FAST_BLINDING,
 *    BPG_FLAG_WITNESS_ON_DEVICE, BPG_FLAG_FORCE_LATE_FOLD and a sharded context (world > 1) return BPG_E_ARG.  Witness
 *    buffers are host pointers.
 *  - The batched path neither uses nor consumes bpg_r1cs_prove_prefetch hints; a delegated proof behaves as bpg_r1cs_prove.
 *  - Secrets (witness, s_L / s_R, l / r vectors, blindings) are wiped on the device and on the host before the call returns.
 *  - count has no upper limit: the batch is split internally into passes of bounded scratch, with unchanged bytes. */
int bpg_r1cs_prove_batch(bpg_ctx *ctx, size_t count, bpg_circuit *const *circuits, const uint8_t *const *labels,
                         const size_t *label_lens, const uint8_t *const *aL, const uint8_t *const *aR, const uint8_t *const *aO,
                         const uint8_t *const *v, const uint8_t *const *v_blinding, const uint8_t *ext_rng32, unsigned flags,
                         uint8_t *const *V_out, uint8_t *const *proofs, const size_t *proof_caps, size_t *proof_lens);
/* Verifier::new(label) + commit(V_i)* + (constraints) + verify(&proof,&pc_gens,&bp_gens)  [ext; verifier.rs:51-53,90].
 * *accept = 1 for Ok(()), 0 for Err(VerificationError | FormatError); the return value only reports library errors. */
int bpg_r1cs_verify(bpg_ctx *ctx, bpg_circuit *c, const uint8_t *label, size_t label_len, const uint8_t *V32,
                    const uint8_t *proof, size_t proof_len, const uint8_t ext_rng32[32], unsigned flags, int *accept);

/* Batch verification (SURVEY 8 f-4): accept[i] = what bpg_r1cs_verify returns for proof i.  The proofs are combined
 * with random weights into ONE fixed-base multiscalar multiplication over the resident generators plus one
 * variable-base launch over all proofs' own points; a failing combination is bisected until the invalid proofs are
 * isolated, so verdicts equal one-by-one verification.  ext_rng32 = count x 32 bytes (one thread_rng stand-in per proof):
 * it MUST be fresh secret randomness (the reference draws it from thread_rng inside Verifier::verify).  The combination
 * weights are derived from every proof's label, commitments and full proof bytes together with ext_rng32, so they are
 * bound to the statements being checked and cannot be anticipated by the provers. */
int bpg_r1cs_verify_batch(bpg_ctx *ctx, size_t count, bpg_circuit *const *circuits, const uint8_t *const *labels,
                          const size_t *label_lens, const uint8_t *const *V32, const uint8_t *const *proofs,
                          const size_t *proof_lens, const uint8_t *ext_rng32, unsigned flags, int *accept);

/* Merlin transcript (host; sequential Keccak, never on the device) exposed for the Rust shim and the tests */
typedef struct bpg_transcript bpg_transcript;
bpg_transcript *bpg_transcript_new(const uint8_t *label, size_t len);
void bpg_transcript_free(bpg_transcript *t);
void bpg_transcript_append(bpg_transcript *t, const uint8_t *label, size_t ll, const uint8_t *msg, size_t ml);
void bpg_transcript_challenge(bpg_transcript *t, const uint8_t *label, size_t ll, uint8_t *out, size_t n);
/* merlin TranscriptRng (the prover's source of blinding factors; Prover::prove behind src/bin/prover.rs:93).  Concurrent
 * provers of one process share a lane-batched Keccak (4 streams per AVX2 / 8 per AVX-512 register file);
 * bpg_host_rng_lanes() reports the width in use (1 = scalar; BPG_RNG_LANES=1 forces it).  bpg_host_rng_draw64 writes
 * count + 1 draws of 64 bytes of TranscriptRng(Transcript(label)).finalize(ext32) after `warm` discarded draws: the
 * first `count` through the service (use_service = 1) or the scalar definition (0), the last one always scalar. */
int bpg_host_rng_lanes(void);
int bpg_host_rng_draw64(const uint8_t *label, size_t label_len, const uint8_t ext32[32], size_t warm, size_t count, int use_service,
                        uint8_t *out);

/* device memory helpers for callers that keep vectors resident (bench, multi-GPU drivers) */
int bpg_dev_alloc(bpg_ctx *ctx, size_t bytes, void **d_ptr);
int bpg_dev_free(bpg_ctx *ctx, void *d_ptr);
int bpg_dev_upload(bpg_ctx *ctx, void *d_dst, const void *h_src, size_t bytes);
int bpg_dev_download(bpg_ctx *ctx, void *h_dst, const void *d_src, size_t bytes);
/* Page-locked host memory for callers that hand large host vectors to bpg_r1cs_prove (a_L, a_R, a_O: 96 bytes per
 * multiplier).  Every entry point accepts ordinary (pageable) host pointers; from a buffer allocated here the upload is one
 * asynchronous DMA at full PCIe rate instead of a staged copy the calling thread has to wait for (the witness of a
 * 2^20-multiplier proof: ~2 ms instead of ~9 ms).  The Rust side would keep its Vec<Scalar> assignment in such a buffer. */
int bpg_host_alloc(bpg_ctx *ctx, size_t bytes, void **h_ptr);
int bpg_host_free(bpg_ctx *ctx, void *h_ptr);

/* timing on the library's own stream: record event slot i (0..15), elapsed milliseconds between two slots
 * (slots 14 / 15 are recorded by bpg_mimc_sponge_batch around its kernel, 12 / 13 by bpg_fold_points around the fold kernel) */
int bpg_event_record(bpg_ctx *ctx, int slot);
int bpg_event_elapsed_ms(bpg_ctx *ctx, int slot_a, int slot_b, float *ms);
/* per-kernel profile of the MSM bucket-accumulation kernel (the dominant kernel): while enabled every launch is
 * (up to the first 64 after enabling) is bracketed by CUDA events; bpg_prof_read returns the number of launches, their summed duration and the summed
 * number of (term, window) pairs they accumulated since the last enable */
int bpg_prof_enable(bpg_ctx *ctx, int on);
int bpg_prof_read(bpg_ctx *ctx, uint64_t *launches, double *ms_total, uint64_t *pairs_total);
/* the same, launch by launch (up to cap): duration in ms and sorted pairs of each timed k_msm_accumulate launch; returns the count */
long bpg_prof_read_launches(bpg_ctx *ctx, float *ms, uint32_t *pairs, size_t cap);

/* integer-pipe microbenchmark: runs `iters` dependent field multiplications per thread over a full-chip grid and
 * returns elapsed milliseconds (CUDA events) and the number of 32x32->64 multiply-accumulates executed */
int bpg_bench_imad(bpg_ctx *ctx, int iters, float *ms, double *mac32);

/* single-warp latency (SM cycles per operation) of dependent operations: [0] fe_mul [1] ge_add [2] ge_add interleaved
 * [3] ge_dbl [4] ge_dbl interleaved [5] mixed add [6] mixed add interleaved [7] four interleaved fe_mul */
int bpg_bench_latency(bpg_ctx *ctx, int iters, double cycles_per_op[8]);

#ifdef __cplusplus
}
#endif
#endif
