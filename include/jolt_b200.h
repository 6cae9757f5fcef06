/* jolt_b200.h - C ABI of the B200 (sm_100a) backend for the a16z/jolt prover hot path.
 *
 * The reference (a16z/jolt @ ff9f8c13) has no FFI today: its compute seam is a set of Rust
 * traits. Each entry point below names the reference interface it replaces (file:line under
 * /root/reference); INTEGRATION.md shows the Rust-side binding a maintainer would add.
 *
 * Conventions (specs/clean-slate-prover.md:565-591):
 *  - Field elements are 4 x uint64_t little-endian Montgomery limbs (a * 2^256 mod p), exactly
 *    `Fr::inner_limbs()` (crates/jolt-field/src/bn254/mod.rs:33-42). Every output is canonical
 *    (fully reduced, < p).
 *  - G1 points cross the ABI as affine (x, y) = 8 limbs over Fq (Montgomery); the identity is
 *    x = y = 0. Jacobian inputs/outputs are 12 limbs (X, Y, Z), identity Z = 0
 *    (`Bn254G1` = repr(transparent) G1Projective, crates/jolt-crypto/src/ec/bn254/mod.rs:17-24).
 *  - Host buffers are borrowed for the duration of the call. Device state lives in a context
 *    (one per ProofSession, crates/jolt-kernels/src/backend.rs:283-286) and is freed with it.
 *  - Every function returns a jb_status; nothing unwinds or aborts across the ABI
 *    (maps to KernelError / SumcheckError, crates/jolt-kernels/src/error.rs:80-89).
 *  - A context serialises its calls with an internal mutex; distinct contexts are independent
 *    (Rayon threads call msm concurrently, crates/jolt-hyperkzg/src/scheme.rs:141-145).
 *  - There is NO CPU fallback: without a CUDA device every compute entry point returns
 *    JB_ERR_NO_DEVICE.
 */
#ifndef JOLT_B200_H
#define JOLT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum jb_status {
    JB_OK = 0,
    JB_ERR_NO_DEVICE = 1,    /* no CUDA device / driver */
    JB_ERR_CUDA = 2,         /* a CUDA call failed (see jb_last_error) */
    JB_ERR_INVALID = 3,      /* KernelError::InvariantViolation: bad handle, length, order ... */
    JB_ERR_OOM = 4,          /* device allocation failed (recoverable at plan time) */
    JB_ERR_ROUND_CHECK = 5,  /* SumcheckError::RoundCheckFailed: s(0)+s(1) != previous_claim */
    JB_ERR_UNSUPPORTED = 6,  /* KernelError::Unsupported */
    JB_ERR_LENGTH = 7        /* msm: bases/scalars length mismatch (mod.rs:200-204) */
} jb_status;

/* BindingOrder, crates/jolt-poly/src/lib.rs (HighToLow pairs (i, i+half); LowToHigh (2i, 2i+1)). */
typedef enum jb_order { JB_HIGH_TO_LOW = 0, JB_LOW_TO_HIGH = 1 } jb_order;

/* Element encodings. JB_SCALAR_FR = 4 x u64 Montgomery limbs. The others are the primitive integer columns
 * the reference keeps compact - `Polynomial<T>` (crates/jolt-poly/src/dense.rs:22-142), legacy
 * MultilinearPolynomial::{U8Scalars..I128Scalars} (crates/jolt-prover-legacy/src/msm/mod.rs:27-79) - as
 * native little-endian arrays (u128/i128: 16 bytes, low half first; bool columns are U8 with values 0/1).
 * Their field value is Ring::from_u64/from_i64/from_u128/from_i128
 * (crates/jolt-field/src/bn254/mod.rs:265-298): v mod r, negatives as r - |v|. */
typedef enum jb_scalar_kind {
    JB_SCALAR_FR = 0,
    JB_SCALAR_U8 = 1,
    JB_SCALAR_U16 = 2,
    JB_SCALAR_U32 = 3,
    JB_SCALAR_U64 = 4,
    JB_SCALAR_U128 = 5,
    JB_SCALAR_I64 = 6,
    JB_SCALAR_I128 = 7,
    JB_SCALAR_S64 = 8,  /* array of jb_s64 */
    JB_SCALAR_S128 = 9  /* array of jb_s128 */
} jb_scalar_kind;

/* Sign-magnitude integers: jolt_field::signed::S64 / S128 = SignedBigInt<1> / SignedBigInt<2>
 * { magnitude: Limbs<N>, is_positive: bool } (crates/jolt-field/src/signed.rs:25-32), the scalars of the legacy
 * msm_s64 / msm_s128 (crates/jolt-prover-legacy/src/msm/mod.rs:140-158) and of MultilinearPolynomial::S128Scalars
 * (poly/multilinear_polynomial.rs:33). The Rust struct is not repr(C); these are the records the adapter passes
 * (a #[repr(C)] mirror; on x86-64 / aarch64 rustc lays SignedBigInt<N> out exactly like this). Field value:
 * +-magnitude mod r; "zero is not canonicalized" (signed.rs:16-17): a zero magnitude with either sign is 0. */
typedef struct jb_s64 { uint64_t magnitude; uint8_t is_positive; uint8_t pad[7]; } jb_s64;       /* 16 bytes */
typedef struct jb_s128 { uint64_t magnitude[2]; uint8_t is_positive; uint8_t pad[7]; } jb_s128;  /* 24 bytes */

typedef struct jb_ctx jb_ctx;       /* ~ ProofSession: device pools + stream */
typedef struct jb_member jb_member; /* ~ Box<dyn SumcheckKernel>: a ProveRounds member on device */
typedef uint64_t jb_table;          /* device-resident Polynomial<Fr> / DensePolynomial<Fr> */
typedef uint64_t jb_srs;            /* device-resident affine G1 bases (HyperKZGProverSetup::g1_powers) */

/* ---- library / context ---------------------------------------------------------------- */
const char* jb_version(void);
const char* jb_status_str(int status);
int jb_device_count(void);
/* ProofSession::new - owns a stream and memory pools on `device`. */
int jb_ctx_create(int device, jb_ctx** out);
/* Same, but enqueues on a caller-owned cudaStream_t (e.g. torch's current stream). */
int jb_ctx_create_on_stream(int device, void* cuda_stream, jb_ctx** out);
void jb_ctx_destroy(jb_ctx* ctx);
const char* jb_last_error(jb_ctx* ctx);
int jb_ctx_synchronize(jb_ctx* ctx);
/* 1: members compute s(1) and check every round against the claim (reference tier); 0 (default):
 * s(1) = claim - s(0) (optimized tier). Proof-invariant: both yield identical round polynomials. */
int jb_ctx_set_verify_rounds(jb_ctx* ctx, int on);
/* Kernel launches issued by this context so far (bench.py's gpu_launches claim). */
uint64_t jb_ctx_launch_count(jb_ctx* ctx);

/* ---- tables: Polynomial<Fr>::new (crates/jolt-poly/src/dense.rs:35-60),
 *      DensePolynomial::new (crates/jolt-prover-legacy/src/poly/dense_mlpoly.rs:27-39) --------- */
int jb_table_upload(jb_ctx* ctx, const uint64_t* mont_limbs, size_t len, jb_table* out);
int jb_table_alloc(jb_ctx* ctx, size_t len, jb_table* out);
/* Borrow caller-owned device memory (len * 32 bytes, 32-byte aligned); never freed by the context. */
int jb_table_wrap_device(jb_ctx* ctx, void* device_ptr, size_t len, jb_table* out);
int jb_table_len(jb_ctx* ctx, jb_table t, size_t* len);
int jb_table_device_ptr(jb_ctx* ctx, jb_table t, void** device_ptr);
int jb_table_download(jb_ctx* ctx, jb_table t, uint64_t* out_limbs, size_t len);
int jb_table_clone(jb_ctx* ctx, jb_table t, jb_table* out);
int jb_table_free(jb_ctx* ctx, jb_table t);

/* Polynomial::bind_with_order (crates/jolt-poly/src/dense.rs:180-263); legacy
 * DensePolynomial::bind / bind_parallel (dense_mlpoly.rs:71-83). Halves the table.
 * `r` = Montgomery limbs of the challenge; limbs [0,0,lo,hi] (the 125-bit MontU128Challenge,
 * crates/jolt-prover-legacy/src/field/challenge/mont_ark_u128.rs:28-34) take the half-cost path. */
int jb_table_bind(jb_ctx* ctx, jb_table t, const uint64_t r[4], int order);
/* Compact tables. upload_small: a host array of `len` primitive integers (kind != JB_SCALAR_FR) becomes a
 * field table, promoted on the device (F::from(T), dense.rs:129-142): 1-16 bytes per entry cross PCIe
 * instead of 32. bind_small: Polynomial<T>::bind_to_field (dense.rs:129-142; the reference folds
 * HighToLow, both orders are offered) - the compact table folded under `r` straight into a NEW field table
 * of len/2 entries, out[i] = F(lo) + r * (F(hi) - F(lo)). Values identical to promoting then binding. */
int jb_table_upload_small(jb_ctx* ctx, const void* values, size_t len, int kind, jb_table* out);
int jb_table_bind_small(jb_ctx* ctx, const void* values, size_t len, int kind, const uint64_t r[4], int order,
                        jb_table* out);

/* EqPolynomial::evals(r, scaling_factor) (crates/jolt-poly/src/eq.rs:221-231): 2^nvars entries,
 * r[0] <-> most-significant index bit. scale_or_null == NULL means 1. */
int jb_eq_evals(jb_ctx* ctx, const uint64_t* r, size_t nvars, const uint64_t* scale_or_null, jb_table* out);
/* EqPolynomial::evals_for_aligned_block (eq.rs:238-263): the per-GPU slice of a sharded eq table. */
int jb_eq_evals_aligned_block(jb_ctx* ctx, const uint64_t* r, size_t nvars, size_t start_index,
                              size_t block_size, jb_table* out);

/* ---- sumcheck member: ProveRounds (crates/jolt-sumcheck/src/prover.rs:52-72) for the
 *      product-of-m-tables relation, degree m (naive.rs:241-316; tests/roundtrip.rs:26-97) ------- */
/* Takes ownership of the m tables (all the same power-of-two length). m in 1..8 (5..8: the wide product pass, one
 * launch per round; see jb_scheduler_create for the degree the scheduler takes). */
int jb_member_create(jb_ctx* ctx, const jb_table* tables, size_t m, int order, jb_member** out);
/* Sum-of-products member: ProveRounds for  sum_x sum_{k < terms} prod_{j < factors} f_{k * factors + j}(x),
 * degree = factors, over factors * terms dense tables (term k owns tables [k * factors, (k + 1) * factors)); every
 * table is bound by every challenge (bind_all, crates/jolt-kernels/src/optimized/support.rs). This is the shape of the
 * reference's optimized claim-reduction kernels after paired-eq fusion - e.g. IncClaimReduction's summand
 * A * RamInc + B * RdInc (crates/jolt-kernels/src/optimized/inc_claim_reduction.rs:47-203: factors = 2, terms = 2,
 * tables {A, RamInc, B, RdInc}); term weights are folded into one table of the term, as the reference folds gamma
 * into A and B. Built shapes: terms = 1 with factors 1..8 (== jb_member_create) and factors = 2, terms = 2.
 * jb_member_final_evals returns the factors * terms bound values in table order. */
int jb_member_create_sop(jb_ctx* ctx, const jb_table* tables, size_t factors, size_t terms, int order, jb_member** out);
int jb_member_num_tables(jb_member* mem, size_t* tables);
jb_ctx* jb_member_context(jb_member* mem);
int jb_member_num_rounds(jb_member* mem, size_t* rounds);
int jb_member_degree(jb_member* mem, size_t* degree);
/* prove_round(bind, round, previous_claim): binds `bind_or_null` (NULL on the first active round)
 * and returns the evaluations s(0..degree) (degree+1 elements) of the round polynomial, fused in
 * one pass over the tables. With a claim, s(1) is derived as previous_claim - s(0) (the optimized
 * tier's convention, jolt-kernels/src/optimized/support.rs:450-460) unless
 * jb_ctx_set_verify_rounds(ctx, 1) is in force, in which case every point is computed and
 * JB_ERR_ROUND_CHECK is returned if s(0)+s(1) != previous_claim (the reference tier,
 * naive.rs:301-308). Without a claim every point is computed and nothing is checked. */
int jb_member_prove_round(jb_member* mem, const uint64_t* bind_or_null, size_t round,
                          const uint64_t* previous_claim_or_null, uint64_t* out_evals);
/* finish_rounds(bind): the terminal bind. */
int jb_member_finish_rounds(jb_member* mem, const uint64_t bind[4]);
/* The m fully bound table values (SumcheckKernel::output_claims, kernel.rs:72-126). */
int jb_member_final_evals(jb_member* mem, uint64_t* out_m_elems);
/* Split-eq member (SURVEY 8f rank 2): ProveRounds for sum_x eq(w, x) * prod_j f_j(x), degree m + 1, without
 * ever materialising or binding the eq table - GruenSplitEqPolynomial / TensorEqTable
 * (crates/jolt-poly/src/split_eq.rs:10-447): each round's sweep is weighted by E_out (x) E_in over the
 * not-yet-current variables (two ~sqrt(N) tables), the current variable's linear factor and the hint
 * s(0)+s(1) = previous_claim complete the round polynomial on the host (gruen_poly_from_evals, :404-437).
 * w = nvars elements, w[0] <-> most significant index bit; both binding orders (LowToHigh: prefix tables
 * evals_cached, split_eq.rs:208-232; HighToLow: suffix tables evals_cached_rev, :233-257); m in 1..8, so the degree is at
 * most 9 and out_evals of jb_member_prove_round takes m + 2 elements; the running claim
 * is mandatory in prove_round. Round polynomials equal those of the (m+1)-table product member over the
 * materialised eq table. jb_eq_member_scalar returns scale * eq(w, r) after the rounds. */
int jb_eq_member_create(jb_ctx* ctx, const jb_table* tables, size_t m, const uint64_t* w, size_t nvars,
                        const uint64_t* scale_or_null, int order, jb_member** out);
int jb_eq_member_scalar(jb_member* mem, uint64_t out[4]);
/* Multi-GPU: like prove_round but leaves this rank's partial sums - the kernel values s(0), [s(1) unless
 * skip_t1], s(2), .., s(m-1), s(inf) in the order jb_round_evals_from_kernel_values documents - on the device as
 * count x 8 uint64 lanes, each holding one 32-bit limb (exact under ncclSum over <= 2^32 ranks); the caller
 * all-reduces that buffer, calls jb_partials_finalize and then jb_round_evals_from_kernel_values. No round check.
 * Members of 1..4 tables only (JB_ERR_UNSUPPORTED otherwise). */
int jb_member_prove_round_partials(jb_member* mem, const uint64_t* bind_or_null, size_t round, int skip_t1,
                                   void* device_lanes_out);
int jb_partials_finalize(jb_ctx* ctx, const void* device_lanes, size_t count, uint64_t* out_elems);
/* The host half of the above (carry-propagate + fold mod r) on `count` x 8 host lanes; needs no device. */
int jb_lanes_reduce_host(const uint64_t* lanes, size_t count, uint64_t* out_elems);
/* The host half of a resident-kernel round (needs no device): `count` x 17 u64 lanes, each value the block-summed
 * UNREDUCED accumulator sum_y a_y b_y over Montgomery operands (lane w = sum of the 32-bit limbs of weight 2^(32 w))
 * -> canonical (sum) R^-1 mod r. The O(degree) serial tail of a round - carry propagation and the Montgomery
 * reduction of a 544-bit sum - takes one CPU core ~0.2 us and one GPU lane ~2 us, and it sits on the latency path
 * of every round, so the resident kernel hands it to the host (as the reference's host keeps interpolation). */
int jb_wide_lanes_reduce_host(const uint64_t* lanes, size_t count, uint64_t* out_elems);
/* The host half of a round (needs no device). The round kernels emit, for a product of m tables,
 *   s(0), [s(1) unless skip_t1], s(2), .., s(m-1), s(inf)      (m >= 2; s(inf) = the leading coefficient)
 *   s(0), [s(1) unless skip_t1]                                (m == 1)
 * and this rebuilds the m + 1 evaluations s(0), .., s(m) the interpolation takes: s(1) = claim - s(0) when it was
 * skipped (round_poly_from_skipped_evals, crates/jolt-kernels/src/optimized/support.rs:450-460) and s(m) from the
 * leading coefficient (the evaluation-at-infinity trade of UnivariatePoly::from_evals_toom). With a claim and
 * skip_t1 == 0 the round check s(0) + s(1) == claim is applied (JB_ERR_ROUND_CHECK). jb_member_prove_round calls
 * exactly this on the values the device published. */
int jb_round_evals_from_kernel_values(int m, int skip_t1, const uint64_t* kernel_values, const uint64_t* claim_or_null,
                                      uint64_t* out_evals);
/* Copies table j of a member (current, possibly partly bound contents) to caller device memory -
 * used to all-gather the shards once they are small (jolt_b200/dist.py). */
int jb_member_export_table(jb_member* mem, size_t j, void* device_dst, size_t cap_elems, size_t* len_out);
void jb_member_destroy(jb_member* mem);

/* ---- multi-GPU (SURVEY 8e): one process per GPU; the caller owns rendezvous (torch.distributed
 * broadcasts the 128-byte NCCL unique id), the context issues the per-round collectives itself on its
 * stream. libnccl is resolved at run time (pass NULL to use the copy already loaded in the process). */
int jb_comm_unique_id(uint8_t out[128], const char* libnccl_path_or_null);
int jb_comm_init(jb_ctx* ctx, int nranks, int rank, const uint8_t id[128], const char* libnccl_path_or_null);
int jb_comm_destroy(jb_ctx* ctx);
/* Optional, after jb_comm_init: peer-memory exchange buffers (CUDA IPC over NVLink). Each rank exports
 * the 64-byte handle of its buffer, the caller all-gathers them (rank order) and every rank opens them.
 * Sharded members then perform the per-round all-reduce INSIDE the round kernel (the finishing thread
 * stores its lanes into every peer's buffer, waits for the others' and sums) - no NCCL launch per round.
 * If opening fails the NCCL path remains in force. */
int jb_comm_p2p_handle(jb_ctx* ctx, uint8_t out[64]);
int jb_comm_p2p_open(jb_ctx* ctx, const uint8_t* handles_world_x_64);
/* An index-sharded ProveRounds member. `order` fixes the partition that keeps every (lo, hi) pair local
 * (SURVEY 8e): JB_LOW_TO_HIGH pairs (2i, 2i+1) -> this rank's m tables are the CONTIGUOUS block `rank` of the
 * global tables, local[j] = global[rank * n + j]; JB_HIGH_TO_LOW pairs (i, i + half) -> the STRIDED shard,
 * local[j] = global[j * nranks + rank]. It reports log2(local len) + log2(nranks)
 * rounds and is driven by the same jb_member_prove_round / jb_prove_batch as a local member: each early
 * round costs ONE all-reduce of <= 40 u64; when a shard is 2^gather_log long the shards are
 * all-gathered once and every rank finishes the remaining rounds redundantly (identical results on all
 * ranks, identical to the single-GPU member over the global tables). `previous_claim` is the GLOBAL claim.
 * m in 1..4 (JB_ERR_UNSUPPORTED otherwise). */
int jb_sharded_member_create(jb_ctx* ctx, const jb_table* tables, size_t m, int order, size_t gather_log,
                             jb_member** out);

/* ---- device RoundScheduler: jolt_sumcheck::RoundScheduler (crates/jolt-sumcheck/src/prover.rs:106-120), minted per
 * stage by BuildRoundScheduler::build(session) (crates/jolt-kernels/src/backend.rs:64-70, "so a device traversal
 * shares the carry"). "Order and transport are free": a batch round costs ONE host round trip whatever the member
 * count. Homogeneous batches (same shape and order, <= 8 members) are served by ONE resident kernel - launched once,
 * it takes every round's {per-member action, shared challenge} from a mailbox in host-mapped memory and answers
 * with every member's round sums, so no kernel is launched per round; otherwise every active member's pass is
 * enqueued before the first wait (one result slot per member). `work[i].member` indexes the member list given at
 * creation; out_evals receives 8 elements (32 limbs) per work item, the first degree + 1 of them valid. So members
 * of degree at most 7 only: jb_scheduler_create returns JB_ERR_UNSUPPORTED for a product of 8 tables or a split-eq
 * member of 7 or 8 tables (jb_prove_batch then proves the batch's members in declaration order).
 * Results are identical to calling jb_member_prove_round on each item. ------------------------------------------ */
typedef struct jb_scheduler jb_scheduler;
typedef struct jb_round_work {   /* MemberRound, prover.rs:75-92 */
    size_t member;
    size_t round;                /* member-local round */
    int has_bind;                /* 0 exactly on the member's first active round */
    int has_claim;               /* 0: compute every point, check nothing (as jb_member_prove_round without a claim) */
    uint64_t bind[4];
    uint64_t claim[4];
} jb_round_work;
typedef struct jb_finish_work {  /* MemberFinish, prover.rs:94-104 */
    size_t member;
    uint64_t bind[4];
} jb_finish_work;
int jb_scheduler_create(jb_ctx* ctx, jb_member** members, size_t n_members, jb_scheduler** out);
int jb_scheduler_prove_round(jb_scheduler* s, const jb_round_work* work, size_t n_work, uint64_t* out_evals);
int jb_scheduler_finish_rounds(jb_scheduler* s, const jb_finish_work* work, size_t n_work);
void jb_scheduler_destroy(jb_scheduler* s);

/* ---- batched engine: jolt_sumcheck::prove_batch (crates/jolt-sumcheck/src/prover.rs:193-362) over
 *      device members, SequentialRounds traversal. BatchMember = batch.rs:24-71. The transcript stays
 *      with the caller: `absorb` receives each round's batched polynomial (trimmed coefficients, 4
 *      limbs each) and returns the challenge (recorder.absorb_round, recorder.rs:118-130); a non-zero
 *      return aborts. Outputs = ProvedBatch (prover.rs:153-157) + the round polynomials, zero-padded
 *      to max_degree+1 coefficients per round. ---------------------------------------------------- */
typedef struct jb_batch_member {
    uint64_t input_claim[4];
    uint64_t coefficient[4];
    size_t rounds;
    size_t offset;
} jb_batch_member;
typedef int (*jb_absorb_round_fn)(void* user, size_t round, const uint64_t* coeffs, size_t ncoeffs,
                                  uint64_t challenge_out[4]);
int jb_prove_batch(jb_member** members, const jb_batch_member* desc, size_t n_members, size_t max_num_vars,
                   size_t max_degree, const uint64_t claimed_sum[4], int check_member_rounds,
                   jb_absorb_round_fn absorb, void* user, uint64_t* out_challenges, uint64_t out_final_claim[4],
                   uint64_t* out_member_claims, uint64_t* out_round_polys, size_t* out_round_poly_lens);
/* A deterministic stand-in transcript for benches/tests: 125-bit challenge [0,0,lo,hi] from the round
 * polynomial via SplitMix64; `user` -> uint64_t seed. (Fiat-Shamir itself is out of scope.) */
int jb_absorb_round_splitmix125(void* user, size_t round, const uint64_t* coeffs, size_t ncoeffs,
                                uint64_t challenge_out[4]);

/* ---- G1 MSM: JoltGroup::msm (crates/jolt-crypto/src/ec/group.rs:70; impl
 *      ec/bn254/mod.rs:195-212) and kzg_commit (crates/jolt-hyperkzg/src/kzg.rs:15-27) ------- */
/* Upload bases once per ProverSetup (HyperKZGProverSetup::g1_powers, scheme.rs:60-66). */
int jb_srs_upload_affine(jb_ctx* ctx, const uint64_t* xy_limbs, size_t n, jb_srs* out);
/* Jacobian bases as JoltGroup::msm receives them; normalised on device (batch inversion). */
int jb_srs_upload_jacobian(jb_ctx* ctx, const uint64_t* xyz_limbs, size_t n, jb_srs* out);
/* Synthetic bases generated on the device: bases[i] = (i + 1) * base (affine base point). Valid,
 * distinct curve points with a closed form for checking: msm(s) == (sum_i s_i (i+1)) * base. */
int jb_srs_generate_multiples(jb_ctx* ctx, const uint64_t base_xy[8], size_t n, jb_srs* out);
/* Optional, for a fixed SRS (HyperKZGProverSetup lives as long as the prover): builds the table
 * 2^(c w) * bases[i] for every window w (c = window_bits, 0 = choose from the SRS length), W x the SRS in
 * HBM (e.g. 12 x 1 GiB at 2^24). MSMs over this handle with n >= 2^(c-4) then use ONE bucket set for
 * all windows: wider windows (fewer bucket additions), no per-window reduction, no 2^(c w) doubling
 * chains. Results are identical group values. JB_ERR_OOM leaves the handle usable on the plain path. */
int jb_srs_precompute(jb_ctx* ctx, jb_srs s, int window_bits);
int jb_srs_len(jb_ctx* ctx, jb_srs s, size_t* n);
int jb_srs_download_affine(jb_ctx* ctx, jb_srs s, uint64_t* out_xy, size_t n);
int jb_srs_free(jb_ctx* ctx, jb_srs s);
/* sum_i scalars[i] * bases[offset + i], i < n; scalars = host Montgomery limbs (any Fr value, the
 * canonical integer is used, mod.rs:208). Result: a Jacobian representative X, Y, Z of the group
 * value (x = X/Z^2, y = Y/Z^3; Z = 0 for the identity) - `Bn254G1` equality is projective, so no
 * normalisation is needed (or paid for) at the boundary. n == 0 -> identity (group_laws.rs:143-146);
 * offset + n > srs length -> JB_ERR_LENGTH (the reference panics, mod.rs:200-204). */
int jb_msm_g1(jb_ctx* ctx, jb_srs bases, size_t offset, const uint64_t* scalars, size_t n, uint64_t out_xyz[12]);
/* Small-scalar MSM: VariableBaseMSM::msm_u8/u16/u32/u64/u128/i64/i128/s64/s128 and the U8Scalars..I64Scalars arms of
 * VariableBaseMSM::msm (crates/jolt-prover-legacy/src/msm/mod.rs:27-150; msm_binary = JB_SCALAR_U8 with
 * values 0/1). `scalars`: host array of n primitive integers of `kind` (not JB_SCALAR_FR). Only
 * ceil(bits / c) windows are formed and the window is sized for the width (one 9-bit window for u8, five
 * 13-bit windows for u64); a negative scalar flips the sign of its digits. Skewed columns (one-hot, binary:
 * every point in one bucket) are cut into up to 16384 chunks per bucket. A JB_SCALAR_U8 column of >= 2^14 entries is
 * dispatched like the reference's U8Scalars arm (mod.rs:35-47, 96-106): all zero -> identity, all <= 1 -> msm_binary
 * (the plain sum of the selected bases, no digits and no sort), else msm_u8. Same result conventions as jb_msm_g1. */
int jb_msm_g1_small(jb_ctx* ctx, jb_srs bases, size_t offset, const void* scalars, size_t n, int kind,
                    uint64_t out_xyz[12]);
/* VariableBaseMSM::batch_msm and batch_msm_univariate (crates/jolt-prover-legacy/src/msm/mod.rs:160-181): `count` MSMs,
 * MSM k over the PREFIX bases[0 .. lens[k]) with the host column scalars[k] of kind kinds[k] (JB_SCALAR_FR = 4 x u64
 * Montgomery limbs per entry: the LargeScalars arm / UniPoly coefficients; otherwise a primitive column as for
 * jb_msm_g1_small). out_xyz: count x 12 limbs. The reference runs them on a Rayon pool; here they are enqueued back to
 * back on the context's stream (each one already fills the device). Any lens[k] > srs length -> JB_ERR_LENGTH before
 * anything runs (the reference panics in the worker, mod.rs:166). */
int jb_msm_g1_batch(jb_ctx* ctx, jb_srs bases, size_t count, const void* const* scalars, const size_t* lens,
                    const int* kinds, uint64_t* out_xyz);
/* Row-batched MSM: `rows` MSMs of `row_width` terms each against the SAME bases[0 .. row_width), scalars row-major
 * (row r = scalars[r * row_width ..), kind as above, JB_SCALAR_FR allowed) - the tier-1 row commitments of a Dory
 * matrix commitment: DoryScheme::feed / feed_u64 / feed_i128 push one row MSM per chunk and feed_i128_rows_with maps
 * msm_i128 over the windows of a batch on a Rayon pool (crates/jolt-dory/src/streaming.rs:53-70, 113-152, 154-201).
 * Here all the rows go through ONE pass of the pipeline: digits, one scan, one scatter and one bucket accumulation
 * over (row, bucket) sets of 8-bit shared windows (the 2^(8w) * P_i table of the first row_width bases is built on
 * first use and kept with the SRS handle), so a 4096 x 4096 matrix costs one launch sequence, not 4096.
 * out_xyz: rows x 12 limbs (Jacobian, conventions of jb_msm_g1). row_width > srs length -> JB_ERR_LENGTH. */
int jb_msm_g1_rows(jb_ctx* ctx, jb_srs bases, const void* scalars, size_t rows, size_t row_width, int kind,
                   uint64_t* out_xyz);
/* Same with the scalars already on the device (a table, e.g. a folded HyperKZG polynomial). */
int jb_msm_g1_table(jb_ctx* ctx, jb_srs bases, size_t offset, jb_table scalars, size_t n, uint64_t out_xyz[12]);

/* Batch affine addition: batch_g1_additions_multi_affine (crates/jolt-crypto/src/ec/bn254/batch_addition.rs:53-150),
 * the one-hot / binary column path of Dory's tier-1 commitments (crates/jolt-dory/src/streaming.rs:68,128,152,201).
 * Set s is indices[set_offsets[s] .. set_offsets[s + 1]) into `bases`; out_xy receives one AFFINE point per set
 * (8 limbs, identity = zeros for an empty set; a singleton is its base). Every level halves the sets by pairwise
 * affine additions that share batch inversions. Precondition as in the reference: the two points of a pair have
 * distinct x (no repeated or opposite points); a violating pair yields the reference's unchecked garbage for that
 * pair only (zero denominators are skipped by the batch inversion, as ark_ff::batch_inversion does).
 * Indices out of bounds -> JB_ERR_INVALID (the reference documents them as a precondition). */
int jb_g1_batch_add(jb_ctx* ctx, jb_srs bases, const uint64_t* set_offsets, const uint32_t* indices, size_t nsets,
                    uint64_t* out_xy);

/* Multi-GPU MSM (SURVEY 8e): this rank's share of the terms (its own srs handle and host scalars); one
 * all-gather of the G partial points (96 B each) and a local sum give every rank the same total.
 * Needs jb_comm_init. */
int jb_msm_g1_sharded(jb_ctx* ctx, jb_srs bases, size_t offset, const uint64_t* scalars, size_t n, uint64_t out_xyz[12]);
/* Same with a raw device pointer to n Montgomery scalars (32-byte aligned). */
int jb_msm_g1_device(jb_ctx* ctx, jb_srs bases, size_t offset, const uint64_t* device_scalars, size_t n,
                     uint64_t out_xyz[12]);

/* ---- HyperKZG prover side: HyperKZGScheme::open (crates/jolt-hyperkzg/src/scheme.rs:122-158) with
 *      fold_polynomials (scheme.rs:88-114) and kzg_open_batch (kzg.rs:69-126) on the device. commit is
 *      jb_msm_g1_table(srs, 0, evals, 2^ell) (kzg.rs:15-27). `point` = ell elements; evals = 2^ell
 *      entries; the SRS must hold >= 2^ell bases. The transcript stays with the caller:
 *        challenge_r(user, com, ell-1, r_out)  after the ell-1 intermediate commitments (Jacobian, 12 limbs each)
 *        challenge_q(user, v, ell, q_out)      after the evaluations v[t][j] = f_j(u_t), u = [r, -r, r^2]
 *      Outputs: com[(ell-1)][12], w[3][12] (Jacobian representatives), v[3][ell][4]. --------------------- */
typedef int (*jb_hkzg_challenge_r_fn)(void* user, const uint64_t* com_xyz, size_t ncom, uint64_t r_out[4]);
typedef int (*jb_hkzg_challenge_q_fn)(void* user, const uint64_t* v, size_t ell, uint64_t q_out[4]);
int jb_hyperkzg_open(jb_ctx* ctx, jb_srs srs, jb_table evals, const uint64_t* point, size_t ell,
                     jb_hkzg_challenge_r_fn challenge_r, jb_hkzg_challenge_q_fn challenge_q, void* user,
                     uint64_t* out_com, uint64_t* out_w, uint64_t* out_v);

/* ---- raw element-wise ops (parity harness for bn254_differential.rs:75-99) -----------------
 * field: 0 = Fr, 1 = Fq; op: 0 add, 1 sub, 2 mul, 3 mul-by-[0,0,lo,hi], 4 neg(a), 5 square(a) (b ignored
 * for 4 and 5 but must be a valid buffer). Host buffers. */
int jb_vec_op(jb_ctx* ctx, int field, int op, const uint64_t* a, const uint64_t* b, uint64_t* out, size_t n);

/* ---- observability (specs/clean-slate-prover.md:585-587 asks device backends for device-event
 * timing): when enabled, launches of the streaming kernels over >= min_items items are bracketed
 * by CUDA events on the context's stream. collect() synchronises and drains them.
 * kind: 0 fused bind+eval, 1 bind, 2 eval-only, 3 eq, 4 msm bucket accumulation. */
/* out[0] = ns the host spent waiting for round results since the last call, out[1] = number of waits. */
int jb_ctx_diag(jb_ctx* ctx, double out[4]);
/* Per round of the last completed resident-kernel run (<= 64 rounds), 8 values each: device %globaltimer (ns) when
 * the command was decoded and when the last block had folded the round's sums; host CLOCK_MONOTONIC (ns) when the
 * command was posted and when the answer was seen; device: block 0 done with its passes, block 0 arrived, the last
 * block knew it was last, spare. The two clocks are unrelated: use differences. */
int jb_ctx_run_log(jb_ctx* ctx, uint64_t* out, size_t cap_rounds, size_t* rounds);
int jb_ctx_timing_enable(jb_ctx* ctx, int on, uint64_t min_items);
int jb_ctx_timing_collect(jb_ctx* ctx, int* kinds, uint64_t* items, int* m, double* ms, size_t cap, size_t* count);

/* ---- diagnostics (no reference counterpart): sustained Montgomery-product rate of the integer
 * pipes, used for the ALU ceiling quoted beside the HBM roofline in DESIGN.md.
 * variant: 0 full product, 1 product by a [0,0,lo,hi] challenge, 2 add/sub. Giga-ops/s out. */
int jb_diag_mul_throughput(jb_ctx* ctx, int field, int variant, int iters, int blocks, double* out_gops);

#ifdef __cplusplus
}
#endif
#endif /* JOLT_B200_H */
