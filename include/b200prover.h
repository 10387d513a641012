/* libb200prover — C ABI of the B200-native proving backend for the PlonK prover behind
 * renegade-fi/renegade's crates/circuits.
 *
 * This is the drop-in boundary (SURVEY.md §8(b)).  The reference has no FFI for this path: its
 * prover calls Rust crates directly.  Each entry point below names the Rust call it replaces;
 * INTEGRATION.md shows the `extern "C"` block and the safe wrappers a maintainer adds in a new
 * `gpu-prover` shim crate (the existing crates deny `unsafe`: circuit-types/src/lib.rs:4).
 *
 * Conventions
 *   - plain pointers and sizes only; every handle is opaque and owned by the library;
 *   - caller owns all host buffers; the library never keeps a caller pointer past return;
 *   - return 0 on success, negative B200_ERR_* otherwise; never throws, never aborts;
 *     b200_last_error() returns a thread-local message for the last failure;
 *   - field element = 4 x uint64 little-endian limbs (32 bytes).  "Montgomery" = a * 2^256 mod p,
 *     exactly ark-ff's in-memory `Fp256<MontBackend>`; "canonical" = ark-ff `BigInt<4>`;
 *   - G1 affine point = x || y, 64 bytes, Montgomery — one record of the reference's SRS file
 *     (crates/circuits/circuit-types/src/primitives/srs.rs:172-182) and the payload of
 *     `Commitment(G1Affine)`; the identity is flagged separately (and stored as 64 zero bytes);
 *   - a context serialises the calls made on it; use one context per worker thread (rayon
 *     workers in native_proof_manager.rs:187-192) or per GPU for concurrency.
 *   - there is no CPU fallback: without a CUDA device every entry point fails with
 *     B200_ERR_NO_DEVICE.
 */
#ifndef B200PROVER_H
#define B200PROVER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ERR_INVALID (-1)      /* bad argument */
#define B200_ERR_CUDA (-2)         /* CUDA runtime failure (message has the call) */
#define B200_ERR_NOMEM (-3)
#define B200_ERR_FORMAT (-4)       /* malformed .ptau */
#define B200_ERR_NOT_ON_CURVE (-5) /* srs.rs:179 "point not on curve" */
#define B200_ERR_NO_DEVICE (-6)
#define B200_ERR_UNSATISFIED (-7)  /* PlonkError::WrongQuotientPolyDegree: witness does not satisfy the circuit */
#define B200_ERR_MAC (-8)          /* collaborative prover, authenticated shares: the MAC check failed or malformed data was
                                      received; some party deviated and nothing opened during the call may be used */

typedef struct b200_ctx b200_ctx;     /* one CUDA device + stream + scratch */
typedef struct b200_bases b200_bases; /* device-resident G1 bases + window tables (the SRS) */
typedef struct b200_pk b200_pk;       /* device-resident proving key of one circuit */

/* Flat proof, same field order as the reference's `PlonkProof` / `PlonkProofEvaluations`
 * (crates/relayer-types/types-proofs/src/rkyv_impls/plonk_proof_def.rs:168-222); commitments
 * are affine x||y Montgomery, evaluations Montgomery Fr; plookup_proof is always None. */
typedef struct {
    uint64_t wires_poly_comms[5][8];
    uint64_t prod_perm_poly_comm[8];
    uint64_t split_quot_poly_comms[5][8];
    uint64_t opening_proof[8];
    uint64_t shifted_opening_proof[8];
    uint64_t wires_evals[5][4];
    uint64_t wire_sigma_evals[4][4];
    uint64_t perm_next_eval[4];
} b200_proof;

/* ---- lifecycle ------------------------------------------------------------------------- */
/* device: CUDA ordinal.  Replaces nothing in the reference (it has no device). */
int b200_init(int device, b200_ctx** out);
void b200_shutdown(b200_ctx* ctx);
const char* b200_last_error(void);
/* "libb200prover <version> sm_100a" */
const char* b200_version(void);
/* Kernels launched by the library in this process so far (all contexts, all threads). */
uint64_t b200_kernel_launches(void);
/* Host time, in nanoseconds, the calling threads spent submitting those launches (sum over threads). */
uint64_t b200_launch_host_ns(void);
/* From the second proof of a key on a context, b200_plonk_prove replays each prover round as ONE CUDA graph (same kernels,
 * same order, same bytes out; b200_kernel_launches keeps counting the kernels executed).  b200_graph_launches: graph
 * submissions so far.  b200_ctx_use_graphs(ctx, 0) switches the replay off for a context (default: on, or B200_GRAPHS=0
 * in the environment). */
uint64_t b200_graph_launches(void);
int b200_ctx_use_graphs(b200_ctx* ctx, int on);

/* ---- SRS ------------------------------------------------------------------------------- */
/* Replaces parse_ptau_file / read_ptau_header / read_ptau_section1 / read_ptau_section2
 * (srs.rs:63-141): validates magic "ptau", version 1, 11 sections, the Fq modulus and
 * power >= 17, and returns a pointer INTO `bytes` to the first G1 record and the number of
 * records available in section 2.  Host-only, no device work. */
int b200_srs_parse_ptau(const uint8_t* bytes, size_t len, const uint8_t** g1_records,
                        size_t* n_records);

/* Uploads n affine points (64-byte records) and precomputes their window tables.
 * Replaces building `UnivariateUniversalParams.powers_of_g` (srs.rs:70) / the `commit_key`
 * held by `ProvingKey` (traits.rs:850).  window_bits = 0 lets the library choose the Pippenger window
 * for THROUGHPUT (several MSMs / proofs in flight on the GPU, the prover pool's regime: least multiplier
 * work), 1 for LATENCY (one MSM at a time: shortest dependent chains; e.g. c = 16 instead of 15 at 2^13
 * points), 8..23 fixes it.  The result does not depend on the window.
 * check_on_curve != 0 repeats the reference's `is_on_curve` assertion (srs.rs:178-179) on the
 * device and fails with B200_ERR_NOT_ON_CURVE. */
int b200_bases_load(b200_ctx* ctx, const uint8_t* points64, size_t n, int window_bits,
                    int check_on_curve, b200_bases** out);
/* Same, from points already in device memory (device pointer). */
int b200_bases_load_device(b200_ctx* ctx, const void* d_points64, size_t n, int window_bits,
                           b200_bases** out);
void b200_bases_free(b200_ctx* ctx, b200_bases* bases);
size_t b200_bases_len(const b200_bases* bases);
/* plan[0..3] = window bits c, digits per scalar, physical bucket windows, precomputed tables */
void b200_bases_plan(const b200_bases* bases, int plan[4]);

/* ---- MSM ------------------------------------------------------------------------------- */
/* out = sum_{i<n} scalars[i] * bases[base_off + i].
 * Replaces `VariableBaseMSM::msm_bigint(&bases[..], &scalars[..])` followed by
 * `.into_affine()` as used by jf-primitives `UnivariateKzgPCS::commit` (reached from
 * traits.rs:850,996; proof_linking/intent_only.rs:42-47).  scalars_montgomery = 0: canonical
 * `BigInt<4>` (what msm_bigint takes); 1: Montgomery `Fr` coefficients (what `commit` is
 * handed) — the conversion is fused into digit extraction.  Scalars must be < r. */
int b200_msm(b200_ctx* ctx, const b200_bases* bases, size_t base_off, const uint64_t* scalars,
             size_t n, int scalars_montgomery, uint64_t out_xy[8], int* out_is_identity);
/* Same with the scalars already resident in device memory (device pointer). */
int b200_msm_device(b200_ctx* ctx, const b200_bases* bases, size_t base_off,
                    const void* d_scalars, size_t n, int scalars_montgomery, uint64_t out_xy[8],
                    int* out_is_identity);

/* `batch` MSMs over the same bases in one pass: scalar vector i starts at d_scalars + i*stride
 * (elements), each of n scalars; out_xy receives batch x 64 bytes.  Replaces jf-primitives
 * `UnivariateKzgPCS::batch_commit` (the 5 wire / 5 quotient commitments of a proof). */
int b200_msm_batch_device(b200_ctx* ctx, const b200_bases* bases, size_t base_off,
                          const void* d_scalars, size_t n, size_t stride, unsigned batch,
                          int scalars_montgomery, uint64_t* out_xy, int* out_is_identity);

/* Kept for ABI compatibility, no effect: round 1's running-sum bucket reduction had a latency and a
 * throughput setting; the row/column tree reduction that replaced it has one shape for both uses. */
int b200_msm_tuning(b200_ctx* ctx, int throughput_mode);
/* Device-side phase timing (CUDA events recorded on the context's stream).  enable != 0 turns
 * it on for subsequent MSM calls; out_ms (may be NULL) receives the last call's
 * {total, sort = count+scan+scatter, bucket accumulation, bucket reduction} in ms. */
int b200_msm_timing(b200_ctx* ctx, int enable, float out_ms[4]);

/* Running totals of the bucket-accumulation kernel since the last reset while timing is enabled:
 * out = {milliseconds, (point, scalar) pairs, launches}, every MSM call on this context included
 * (the prover's batched commitments too). */
int b200_msm_timing_totals(b200_ctx* ctx, int reset, double out[3]);

/* Sum of k affine points on the host (combining per-GPU partial MSM results after the NCCL
 * gather; ark-ec `Projective += Affine`). */
int b200_g1_sum_affine(const uint64_t* points_xy, const int* is_identity, size_t k,
                       uint64_t out_xy[8], int* out_is_identity);

/* ---- NTT ------------------------------------------------------------------------------- */
/* In-place transform of n = 2^log_n Montgomery Fr elements, natural order in and out.
 * Replaces Radix2EvaluationDomain::<Fr>::{fft_in_place, ifft_in_place, coset_fft_in_place,
 * coset_ifft_in_place} (ark-poly 0.4.2; coset shift = Fr::GENERATOR = 5; ifft scales by n^-1). */
int b200_ntt(b200_ctx* ctx, uint64_t* data, unsigned log_n, int inverse, int coset);
/* `batch` transforms `stride` elements apart, data in device memory (device pointer). */
int b200_ntt_device(b200_ctx* ctx, void* d_data, unsigned log_n, int inverse, int coset,
                    unsigned batch, size_t stride);
/* Device time (CUDA events around the kernels) of the last b200_ntt_device call, in ms. */
int b200_ntt_last_ms(b200_ctx* ctx, float* out_ms);
/* Radix2EvaluationDomain::group_gen (Montgomery). */
int b200_domain_generator(b200_ctx* ctx, unsigned log_n, uint64_t out[4]);

/* ---- synthetic inputs for benchmarks / parity tests (SURVEY.md §8(d)) ------------------- */
/* element i = SplitMix64(seed) outputs 4i..4i+3 as LE limbs, reduced mod r */
int b200_splitmix_fr_device(b200_ctx* ctx, uint64_t seed, size_t first, size_t n, int montgomery,
                            void* d_out);
/* known-discrete-log bases P_i = a_i * G, a_i = splitmix_fr(seed)[first + i]; 64 B records */
int b200_known_dlog_bases_device(b200_ctx* ctx, uint64_t seed, size_t first, size_t n,
                                 void* d_out);

/* ---- TurboPlonk prover (boundary B2, SURVEY.md §8(b)) ------------------------------------ */
/* Replaces `PlonkKzgSnark::<Bn254>::preprocess(&SYSTEM_SRS, &cs)` (traits.rs:850).
 * The host (Rust: `cs` after finalize_for_arithmetization) hands over the circuit structure:
 *   selectors_evals  13 x n selector values over the domain, column order
 *                    q_lc[0..4] q_mul[0..2] q_hash[0..4] q_o q_c q_ecc (Montgomery);
 *   perm             5n entries: perm[i*n + j] = i'*n + j', the copy-constraint permutation
 *                    over wire positions (column i, row j);
 *   k                the 5 coset representatives `vk.k` (Montgomery);
 *   num_inputs       public-input gates occupy rows 0..num_inputs-1.
 * Selector / sigma polynomials, their commitments (the VerifyingKey contents) and the coset
 * evaluations the quotient needs stay resident on the device.  srs must hold >= n + 3 points. */
int b200_plonk_preprocess(b200_ctx* ctx, const b200_bases* srs, unsigned log_n, size_t num_inputs,
                          const uint64_t* selectors_evals, const uint64_t* perm, const uint64_t* k,
                          b200_pk** out);
/* VerifyingKey commitments: 13 selector + 5 sigma commitments, 64 B each. */
int b200_pk_verifying_key(const b200_pk* pk, uint64_t* selector_comms, uint64_t* sigma_comms);
/* Shape of a key: number of public inputs and log2 of the domain size it was preprocessed for. */
size_t b200_pk_num_inputs(const b200_pk* pk);
unsigned b200_pk_log_n(const b200_pk* pk);
void b200_pk_free(b200_ctx* ctx, b200_pk* pk);

/* Replaces `PlonkKzgSnark::prove_with_link_hint::<_, _, SolidityTranscript>(&mut rng, &circuit,
 * &pk)` (traits.rs:996).  wires: 5 x n wire values (the witness table after synthesis; host
 * or device pointer);
 * pub_inputs: num_inputs values; blinders: the 17 Fr elements the reference draws from its RNG
 * (2 per wire polynomial, 3 for the permutation product, 4 for the quotient split), in draw
 * order, supplied by the caller so both sides can be made deterministic (SURVEY.md §0.3).
 * link_poly (may be NULL): the (n + 2)-coefficient blinded wire-0 polynomial of
 * `LinkingHint.linking_wire_poly`; its commitment is proof->wires_poly_comms[0].
 * challenges (may be NULL): beta, gamma, alpha, zeta, v, u for audit.
 * Fails with B200_ERR_UNSATISFIED where the reference returns WrongQuotientPolyDegree. */
int b200_plonk_prove(b200_ctx* ctx, const b200_pk* pk, const uint64_t* wires,
                     const uint64_t* pub_inputs, const uint64_t* blinders, b200_proof* proof,
                     uint64_t* link_poly, uint64_t* challenges);

/* Flat link proof, field order of mpc-plonk `LinkingProof { quotient_commitment, opening_proof }`
 * (crates/relayer-types/types-proofs/src/mocks.rs:28-30). */
typedef struct {
    uint64_t quotient_commitment[8];
    uint64_t opening_proof[8];
} b200_link_proof;

/* Replaces `PlonkKzgSnark::link_proofs::<SolidityTranscript>(&hint_a, &hint_b, &group_layout,
 * &pk.commit_key)` (circuits-core/src/zk_circuits/proof_linking/intent_only.rs:42-47,
 * intent_and_balance.rs:66-72).  a1 / a2: the two `LinkingHint.linking_wire_poly` coefficient
 * vectors (Montgomery, host or device pointers; lengths may differ), comm1 / comm2 their
 * `linking_wire_comm`; (alignment, offset, size) = mpc-relation `GroupLayout`: the group sits on
 * the roots g^(offset + i), i < size, g the generator of the 2^alignment-th roots of unity.
 * eta (may be NULL) receives the Fiat–Shamir challenge.  Fails with B200_ERR_UNSATISFIED when a1 and a2
 * do not agree on the group (no link proof exists: wrong layout or mismatched witnesses). */
int b200_plonk_link(b200_ctx* ctx, const b200_bases* srs, const uint64_t* a1, size_t len1,
                    const uint64_t* a2, size_t len2, const uint64_t* comm1, const uint64_t* comm2,
                    unsigned alignment, size_t offset, size_t size, b200_link_proof* proof,
                    uint64_t* eta);

/* ---- verification (host only; no device is needed or used) -----------------------------------
 * G2 points are 128-byte records x0 || x1 || y0 || y1 (Montgomery Fq), the layout of the ptau file's
 * G2 section read by srs.rs:185-199: g2_h = `UnivariateUniversalParams.h`, g2_tau_h = `.beta_h`.
 * *accepted = 1 / 0; a malformed (off-curve) proof element is a rejection, not an error. */
/* Replaces `PlonkKzgSnark::<Bn254>::verify::<SolidityTranscript>(&vk, public_inputs, &proof, None)`
 * (traits.rs:1012-1018, reached from `SingleProverCircuit::verify`, traits.rs:1003-1019).  The
 * verifying key is passed flat: domain size 2^log_n, num_inputs, k[5], the 13 selector and 5 sigma
 * commitments (b200_pk_verifying_key). */
int b200_plonk_verify(unsigned log_n, size_t num_inputs, const uint64_t* k, const uint64_t* selector_comms,
                      const uint64_t* sigma_comms, const uint64_t* pub_inputs, const b200_proof* proof,
                      const uint64_t g2_h[16], const uint64_t g2_tau_h[16], int* accepted);
/* Replaces `PlonkKzgSnark::verify_link_proof::<SolidityTranscript>(&comm_a, &comm_b, &link_proof,
 * &group_layout, &open_key)` (proof_linking/intent_only.rs:77-84, `validate_*_link`). */
int b200_plonk_verify_link(const uint64_t* comm1, const uint64_t* comm2, unsigned alignment, size_t offset,
                           size_t size, const b200_link_proof* proof, const uint64_t g2_h[16],
                           const uint64_t g2_tau_h[16], int* accepted);
/* *is_one = [ prod_i e(P_i, Q_i) == 1 ] for k (G1, G2) pairs (64-byte / 128-byte records) with one
 * final exponentiation — the primitive under both verifiers and the reference's SRS unit test
 * (srs.rs:236-266: e(tau^i G, tau H) == e(tau^(i+1) G, H)). */
int b200_pairing_check(const uint64_t* g1_points, const uint64_t* g2_points, size_t k, int* is_one);

/* ---- batch verification (device) --------------------------------------------------------------
 * Many PlonK proofs and link proofs checked in one call: the per-item work (on-curve checks, transcript replay, scalar
 * algebra, the G1 operands of each item's KZG check e(A_j, [tau]_2) == e(B_j, [1]_2)) runs on the context's device; the
 * items are folded with the powers of a Fiat–Shamir weight rho (a Keccak challenge over every item's final transcript
 * state, each link item's opening proof and group layout, and the two G2 records) into ONE two-pair pairing product on
 * the host.  Upstream jellyfish has `PlonkKzgSnark::batch_verify` for this use; the scheme here is this library's own.
 * Verdicts are exactly those of the single verifiers above. */
/* One verifying key of a batch: the flat key of b200_plonk_verify. */
typedef struct {
    unsigned log_n;
    size_t num_inputs;
    const uint64_t* k;              /* 5 x 4 limbs */
    const uint64_t* selector_comms; /* 13 x 8 limbs */
    const uint64_t* sigma_comms;    /* 5 x 8 limbs */
} b200_batch_vk;
/* One PlonK proof of a batch, checked against vks[vk] with num_inputs public inputs. */
typedef struct {
    unsigned vk;
    const uint64_t* pub_inputs;
    size_t num_inputs;
    const b200_proof* proof;
} b200_batch_proof;
/* One link proof of a batch: the arguments of b200_plonk_verify_link. */
typedef struct {
    const uint64_t* comm1;
    const uint64_t* comm2;
    unsigned alignment;
    size_t offset;
    size_t size;
    const b200_link_proof* proof;
} b200_batch_link;
/* *accepted = 1 exactly when every proof and link proof verifies.  item_accepted (may be NULL): n_proofs + n_links
 * flags, proofs first, each equal to what b200_plonk_verify / b200_plonk_verify_link returns for that item alone (an
 * off-curve element, an off-curve key point, or a public-input count other than the key's is a 0, not an error); when
 * the combined check fails, contiguous ranges of items are bisected with the same weights, at most about
 * 2 k log2(n) pairing products for k bad items.  operands (may be NULL): per item the unweighted (A_j, B_j), 2 x 8
 * limbs, affine Montgomery, the identity as zeros (also for an item rejected before its check).
 * pairing_products (may be NULL): how many pairing products the call evaluated.
 * B200_ERR_INVALID: a NULL where data is required, vk >= n_vks, log_n > 28, alignment > 28, size == 0 or an empty
 * batch; B200_ERR_NOT_ON_CURVE: an off-curve G2 point.  Synchronous, on the context's stream; keeps no pointer. */
int b200_plonk_batch_verify(b200_ctx* ctx, const b200_batch_vk* vks, size_t n_vks, const b200_batch_proof* proofs,
                            size_t n_proofs, const b200_batch_link* links, size_t n_links, const uint64_t g2_h[16],
                            const uint64_t g2_tau_h[16], int* accepted, uint8_t* item_accepted, uint64_t* operands,
                            size_t* pairing_products);

/* Wall-clock milliseconds of the last proof's phases on this context: round 1, round 2, round 3
 * (coset NTTs + quotient + split), round 3 commitments, round 4, round 5, then two spare slots. */
int b200_plonk_last_timings(b200_ctx* ctx, float out_ms[8]);

/* ---- prover pool --------------------------------------------------------------------------
 * Device-side counterpart of the reference's `NativeProofManager` thread pool
 * (crates/workers/proof-manager/src/implementations/native_proof_manager.rs:138-201: jobs taken
 * from the queue are handed to rayon workers with `spawn_fifo`, one proof per worker): a FIFO
 * queue drained by `n_workers` host threads, each owning one context on `device`.  Proving keys
 * and SRS tables are shared read-only, so `n_workers` proofs are in flight on one GPU and the
 * latency-bound parts of one overlap the throughput-bound kernels of the others (1 -> 6 workers:
 * 149 -> 269 proofs/s at n = 2^16 on one B200).
 * Ownership: `pub_inputs` and `blinders` are copied at submit; `wires`, the link polynomials and
 * every output buffer stay owned by the caller and must remain valid until the job's ticket has
 * been waited for.  Any thread may submit or wait. */
typedef struct b200_pool b200_pool;
int b200_pool_create(int device, unsigned n_workers, b200_pool** out);
/* Finishes the queued jobs, joins the workers, frees the contexts. */
void b200_pool_destroy(b200_pool* pool);
unsigned b200_pool_workers(const b200_pool* pool);
/* Worker i's context, for set-up calls (b200_bases_load, b200_plonk_preprocess) made while no job
 * is running; keys created on any context of the device can be used by every worker. */
b200_ctx* b200_pool_ctx(b200_pool* pool, unsigned worker);
/* Queue one `b200_plonk_prove(ctx_of_some_worker, pk, wires, pub_inputs, blinders, proof,
 * link_poly, NULL)`; *ticket identifies the job.  num_inputs must equal the key's
 * (b200_pk_num_inputs), else B200_ERR_INVALID. */
int b200_pool_submit_prove(b200_pool* pool, const b200_pk* pk, const uint64_t* wires,
                           const uint64_t* pub_inputs, size_t num_inputs, const uint64_t* blinders,
                           b200_proof* proof, uint64_t* link_poly, uint64_t* ticket);
/* Queue one `b200_plonk_link(...)` (the reference forks its link proofs the same way:
 * native_proof_manager.rs:726-782). */
int b200_pool_submit_link(b200_pool* pool, const b200_bases* srs, const uint64_t* a1, size_t len1,
                          const uint64_t* a2, size_t len2, const uint64_t* comm1, const uint64_t* comm2,
                          unsigned alignment, size_t offset, size_t size, b200_link_proof* proof,
                          uint64_t* ticket);
/* One proof of a bundle, arguments as for b200_pool_submit_prove.  `link_poly` ((2^log_n + 2) x 4 limbs) is required
 * for every proof a link names. */
typedef struct {
    const b200_pk* pk;
    const uint64_t* wires;
    const uint64_t* pub_inputs;
    size_t num_inputs;
    const uint64_t* blinders;
    b200_proof* proof;
    uint64_t* link_poly;
} b200_bundle_proof;
/* One link proof of a bundle: `b200_plonk_link` between the hints of proofs[a] and proofs[b] (in that order) on the
 * group (alignment, offset, size). */
typedef struct {
    unsigned a;
    unsigned b;
    unsigned alignment;
    size_t offset;
    size_t size;
    b200_link_proof* proof;
} b200_bundle_link;
/* Queue a whole proof bundle under ONE ticket: the `n_proofs` proofs run through the pool; when all of them are in,
 * the `n_links` link proofs are forked onto the pool; the ticket completes after the last link proof (or with the
 * first failure).  Replaces the settlement arms of `NativeProofManager::handle_proof_job`
 * (native_proof_manager.rs:526-584) with `compute_private_settlement_link_proofs` (:726-782): e.g. a private match =
 * 5 proofs + 4 links.  The arrays are copied at submit; the buffers they point to stay owned by the caller until
 * the ticket has been waited for. */
int b200_pool_submit_bundle(b200_pool* pool, const b200_bases* srs, const b200_bundle_proof* proofs, size_t n_proofs,
                            const b200_bundle_link* links, size_t n_links, uint64_t* ticket);
/* Blocks until the job is done and returns ITS status (B200_OK or the error the prove/link call
 * returned; b200_last_error() of the waiting thread then holds the job's message).  A ticket can
 * be waited for once. */
int b200_pool_wait(b200_pool* pool, uint64_t ticket);
/* Blocks until the queue is empty and no job is running; returns the oldest failure among the
 * jobs not individually waited for (their tickets are consumed), else B200_OK. */
int b200_pool_wait_all(b200_pool* pool);
/* out = { submitted, completed, failed, queued } */
int b200_pool_stats(b200_pool* pool, uint64_t out[4]);

/* ---- all GPUs of a box behind one object: prover pools + replicated keys -----------------------
 * Whole proofs are independent jobs (SURVEY.md §8(e): replicas, one proof stream per GPU, no communication): a
 * `b200_box` holds one prover pool per device, `b200_box_srs_load` / `b200_box_preprocess` replicate the SRS tables and a
 * proving key on every device (identical results), and every job goes to the device with the fewest unfinished jobs.
 * What ONE host process — the relayer's `NativeProofManager` (native_proof_manager.rs:140-201) — needs to use the
 * whole box.  A ticket encodes its device; tickets are waited for with b200_box_wait. */
typedef struct b200_box b200_box;
typedef struct b200_box_srs b200_box_srs;
typedef struct b200_box_pk b200_box_pk;
int b200_box_create(const int* devices, int n_dev, unsigned workers_per_device, b200_box** out);
void b200_box_destroy(b200_box* box);
int b200_box_devices(const b200_box* box);
/* Device i's pool (b200_pool_* calls work on it directly). */
b200_pool* b200_box_pool(b200_box* box, int i);
int b200_box_srs_load(b200_box* box, const uint8_t* points64, size_t n, int window_bits, int check_on_curve,
                      b200_box_srs** out);
void b200_box_srs_free(b200_box* box, b200_box_srs* srs);
/* b200_plonk_preprocess on every device. */
int b200_box_preprocess(b200_box* box, const b200_box_srs* srs, unsigned log_n, size_t num_inputs,
                        const uint64_t* selectors_evals, const uint64_t* perm, const uint64_t* k, b200_box_pk** out);
int b200_box_pk_verifying_key(const b200_box_pk* pk, uint64_t* selector_comms, uint64_t* sigma_comms);
void b200_box_pk_free(b200_box* box, b200_box_pk* pk);
/* b200_pool_submit_prove on the least-loaded device. */
int b200_box_submit_prove(b200_box* box, const b200_box_pk* pk, const uint64_t* wires, const uint64_t* pub_inputs,
                          size_t num_inputs, const uint64_t* blinders, b200_proof* proof, uint64_t* link_poly,
                          uint64_t* ticket);
/* b200_pool_submit_bundle on the least-loaded device: `pks[i]` is the box key of proofs[i] (the `pk` field of the
 * entries is ignored); a bundle stays on one device. */
int b200_box_submit_bundle(b200_box* box, const b200_box_srs* srs, const b200_box_pk* const* pks,
                           const b200_bundle_proof* proofs, size_t n_proofs, const b200_bundle_link* links,
                           size_t n_links, uint64_t* ticket);
int b200_box_wait(b200_box* box, uint64_t ticket);
/* Index (into the `devices` array) of the device a ticket ran on, -1 for a bad ticket. */
int b200_box_ticket_device(const b200_box* box, uint64_t ticket);

/* ---- multi-GPU: one MSM sharded over the GPUs of a box (SURVEY.md §8(e), boundary B1's
 * `b200_init(const int* devs, int n_dev, ...)`) ----------------------------------------------------
 * Rank g of W owns the points [g n / W, (g + 1) n / W) (b200_shard_range) with resident window tables
 * and gets the matching scalar slice; every GPU runs the whole Pippenger on its shard and contributes
 * ONE group element; the exchange is one `ncclAllGather` of the W 128-byte records over NVLink and a
 * W-term addition on every device, in rank order — the affine result is bit-identical to the
 * single-GPU MSM (G1 addition is associative).  NTT and whole proofs do not shard: use one context /
 * one prover pool per device for those.
 * NCCL is bound at run time (libnccl.so.2); the calls fail with B200_ERR_INVALID when it is absent. */
typedef struct b200_multi b200_multi;             /* contexts + NCCL communicator(s) */
typedef struct b200_multi_bases b200_multi_bases; /* point-range shards of one set of bases */
/* [begin, end) of rank `rank` of `world` over n items (sizes differ by at most one).  Host only. */
void b200_shard_range(size_t n, int rank, int world, size_t* begin, size_t* end);
/* One host process drives all `n_dev` devices (world = n_dev; rank i = devices[i]). */
int b200_multi_init(const int* devices, int n_dev, b200_multi** out);
/* One process per GPU (torchrun): rank 0 makes the id, the host hands it to every rank. */
int b200_nccl_unique_id(uint8_t out[128]);
int b200_multi_init_rank(int device, int rank, int world, const uint8_t unique_id[128], b200_multi** out);
void b200_multi_shutdown(b200_multi* m);
/* NCCL_VERSION_CODE of the library bound at run time. */
int b200_nccl_version(int* version);
int b200_multi_world(const b200_multi* m);
/* devices driven by THIS process (n_dev, or 1 in rank mode), their contexts and global ranks */
int b200_multi_local_devices(const b200_multi* m);
b200_ctx* b200_multi_ctx(b200_multi* m, int local);
int b200_multi_rank(const b200_multi* m, int local);
/* Uploads, for each local device, its range of the n points (the full array is passed) and builds the
 * window tables there; cf. b200_bases_load. */
int b200_multi_bases_load(b200_multi* m, const uint8_t* points64, size_t n, int window_bits,
                          int check_on_curve, b200_multi_bases** out);
/* Synthetic known-discrete-log bases (SURVEY.md §8(d)), generated on each device for its range. */
int b200_multi_bases_known_dlog(b200_multi* m, uint64_t seed, size_t n, int window_bits,
                                b200_multi_bases** out);
void b200_multi_bases_free(b200_multi* m, b200_multi_bases* bases);
size_t b200_multi_bases_len(const b200_multi_bases* bases);
int b200_multi_bases_shard(const b200_multi_bases* bases, int local, size_t* begin, size_t* end);
/* b200_bases_plan of local device `local`'s shard (zeros for an empty shard). */
int b200_multi_bases_plan(const b200_multi_bases* bases, int local, int plan[4]);
/* out = sum_{i<n} scalars[i] * bases[i], n = all points.  `scalars`: the FULL host vector (each local
 * device copies its slice).  Collective: in rank mode every rank must call it; all ranks get the result. */
int b200_multi_msm(b200_multi* m, const b200_multi_bases* bases, const uint64_t* scalars, size_t n,
                   int scalars_montgomery, uint64_t out_xy[8], int* out_is_identity);
/* Same, handing over only the SLICES of the local devices: scalars_local[i] = the scalars of local
 * device i's range — host pointers (scalars_on_device = 0; copied inside the call) or device pointers on
 * that device (1).  NULL is allowed for an empty shard. */
int b200_multi_msm_local(b200_multi* m, const b200_multi_bases* bases, const void* const* scalars_local,
                         int scalars_on_device, int scalars_montgomery, uint64_t out_xy[8], int* out_is_identity);

/* ---- device-vector primitives (Fr, Montgomery, device pointers) -------------------------------
 * The share arithmetic of a collaborative prover (`MultiproverPlonkKzgSnark`, traits.rs:1136) on top of
 * b200_ntt_device / b200_msm_device: element-wise operations, batch inversion of opened values, polynomial
 * evaluation and division by a linear factor.  Each call synchronises the context's stream. */
/* out[i] = a[i] (op) b[i], or a[i] (op) b[0] when b_is_scalar; op 0 add, 1 sub, 2 mul. */
int b200_fr_vec_op(b200_ctx* ctx, int op, const void* d_a, const void* d_b, int b_is_scalar, size_t n, void* d_out);
/* data[i] <- 1 / data[i] in place (0 stays 0). */
int b200_fr_batch_inverse_device(b200_ctx* ctx, void* d_data, size_t n);
/* out = p(z) for the len coefficients at d_coeffs. */
int b200_fr_poly_eval_device(b200_ctx* ctx, const void* d_coeffs, size_t len, const uint64_t z[4], uint64_t out[4]);
/* q = p / (X - z), remainder dropped (len - 1 coefficients written to d_q). */
int b200_fr_poly_div_linear_device(b200_ctx* ctx, const void* d_p, size_t len, const uint64_t z[4], void* d_q);

/* ---- collaborative prover (device) ------------------------------------------------------------
 * `MultiproverPlonkKzgSnark::prove_with_link_hint(&circuit, &pk, fabric)` (traits.rs:1103-1154) for ONE party: each party
 * calls b200_mpc_prove with its own context, its additive shares of the wire table and of the 17 blinders, its
 * preprocessing and a transport to the other parties.  Every party returns the same opened proof and challenges, equal
 * to b200_plonk_prove on the summed wire table and blinders; link_poly_share is this party's share of the linking
 * polynomial (`MpcProofLinkingHint` stays shared).  Opened over the transport: the masked Beaver differences, the masked
 * round-2 denominators den r, partial commitments (summed by the library), the five wire evaluations and z(zeta w), the
 * quotient's coefficients above its degree (zero for a satisfied witness), one masked r q[deg], and the transcript state
 * after the verifying key and the public inputs (every party must agree on it, else B200_ERR_INVALID everywhere).
 * Shares are plain additive shares without MACs (semi-honest parties); the authenticated calls below check them.
 * Every message starts with a 32-byte header (exchange index, payload bytes, two zero words), checked on receipt: the
 * wrong exchange or size is B200_ERR_INVALID.  Any failure after the argument checks calls transport->abort. */
/* all_gather: send `bytes` bytes, receive every party's message in party order (parties * bytes, this party's
 * included); return 0, or a negative code that aborts the proof.  abort (may be NULL): called when this party gives up,
 * so that the others are not left waiting. */
typedef struct {
    int (*all_gather)(void* user, const void* mine, size_t bytes, void* all);
    void (*abort)(void* user);
    void* user;
    int party;   /* 0 .. parties - 1; party 0 adds the public terms */
    int parties; /* >= 2 */
} b200_mpc_transport;
/* Device-resident Beaver triples ([a], [b], [c = a b]) and masks for ONE proof; a second use is B200_ERR_INVALID
 * (reused triples leak the witness).  Layout, n = 2^log_n, m = nc n with nc = 6 (8 below n = 16): round 2 takes
 * R3 = 10 n + sum_{d = 1, 2, .., n/2} (n - d) triples, round 3 the next 26 m, the degree check the last one; the
 * triples [R3 + 2m, R3 + 6m) and [R3 + 11m, R3 + 15m) are squares (c = a^2, b unused).  Masks: n + 1. */
typedef struct b200_mpc_prep b200_mpc_prep;
/* The exact numbers of triples and masks b200_mpc_prove consumes with this key. */
int b200_mpc_prep_size(const b200_pk* pk, size_t* n_triples, size_t* n_masks);
/* This party's shares from the caller's offline phase: a, b, c (n_triples x 4 limbs each), masks (n_masks x 4 limbs);
 * host or device pointers, copied. */
int b200_mpc_prep_load(b200_ctx* ctx, const b200_pk* pk, const uint64_t* a, const uint64_t* b, const uint64_t* c,
                       const uint64_t* masks, b200_mpc_prep** out);
/* INSECURE stand-in for the offline phase, for tests and benchmarks: party p's shares are derived on the device from
 * (seed, p, parties) alone, so no exchange is needed; the last party computes the values and subtracts the other
 * parties' shares.  Anyone who knows the seed knows every triple. */
int b200_mpc_prep_dealer(b200_ctx* ctx, const b200_pk* pk, uint64_t seed, int party, int parties,
                         b200_mpc_prep** out);
void b200_mpc_prep_free(b200_ctx* ctx, b200_mpc_prep* prep);
/* wire_shares: 5 x n (host or device pointer), pub_inputs: the key's num_inputs public values (the same on every party),
 * blinder_shares: 17 (draw order of b200_plonk_prove), proof: the opened proof, link_poly_share (n + 2, may be NULL),
 * challenges (6, may be NULL).  Parties on one device may pass the same key.  B200_ERR_UNSATISFIED on every party when
 * the joint witness does not satisfy the circuit.  A preprocessing with MACs (b200_mpc_prep_*_auth) is B200_ERR_INVALID. */
int b200_mpc_prove(b200_ctx* ctx, const b200_pk* pk, const b200_mpc_transport* transport, b200_mpc_prep* prep,
                   const uint64_t* wire_shares, const uint64_t* pub_inputs, const uint64_t* blinder_shares,
                   b200_proof* proof, uint64_t* link_poly_share, uint64_t* challenges);
/* b200_plonk_link on shares of the two hints (a plaintext hint is passed as its holder's share, zeros elsewhere);
 * comm1 / comm2 are the opened commitments.  Opens the interpolant's coefficients above len - 1 - size (zero when the
 * hints agree on the group, else B200_ERR_UNSATISFIED on every party), the evaluation at eta and partial commitments.
 * The result equals b200_plonk_link on the summed hints. */
int b200_mpc_link(b200_ctx* ctx, const b200_bases* srs, const b200_mpc_transport* transport, const uint64_t* a1_share,
                  size_t len1, const uint64_t* a2_share, size_t len2, const uint64_t* comm1, const uint64_t* comm2,
                  unsigned alignment, size_t offset, size_t size, b200_link_proof* proof, uint64_t* eta);
/* In-process all-gather between the threads of `parties` parties (one b200_mpc_prove call per thread).  After an
 * abort, a failed all_gather or `timeout_ms` without the other parties, every pending and later all_gather of the group
 * fails. */
typedef struct b200_mpc_local_group b200_mpc_local_group;
int b200_mpc_local_group_create(int parties, unsigned timeout_ms, b200_mpc_local_group** out);
/* The transport of `party`; valid while the group lives. */
int b200_mpc_local_group_transport(b200_mpc_local_group* group, int party, b200_mpc_transport* out);
void b200_mpc_local_group_destroy(b200_mpc_local_group* group);
/* The last b200_mpc_prove / b200_mpc_link / b200_mpc_prove_auth / b200_mpc_link_auth on this context: exchanges, bytes
 * sent (headers included), triples used, milliseconds inside all_gather. */
int b200_mpc_last_stats(b200_ctx* ctx, double out[4]);

/* ---- collaborative prover, authenticated shares (device) --------------------------------------------------------
 * The collaborative prover on SPDZ-style authenticated shares, as ark-mpc's `AuthenticatedScalarResult` and
 * `CollaborativePlonkProof::open_authenticated` (circuits-core/src/lib.rs:164-177): each party holds a share alpha_i of
 * a global MAC key alpha (every value Montgomery Fr, 4 limbs), and every shared value x is held as a pair
 * ([x], [alpha x]).  The calls run the same rounds, Beaver levels and messages as b200_mpc_prove / b200_mpc_link on
 * both planes; MAC shares are never sent.  Each opened value x_j leaves this party a record
 * gamma_j = [alpha x_j] - alpha_i x_j.  After the last opening, the parties reveal seeds committed in exchange 0; from
 * them come rho_s, weighting the records as sigma_i = sum_j gamma_j rho_s^(j+1), and rho_p, combining the MAC planes of
 * the committed polynomials into one MSM: Sigma_pt,i = MSM(sum_k rho_p^k [alpha p_k]) - alpha_i sum_k rho_p^k C_k.  The
 * parties commit to (sigma_i, Sigma_pt,i, verdict_i) and reveal them; the call accepts when the sigmas sum to 0, the
 * points to the identity and every verdict is "accept".  A received field element >= r, or a point off the curve
 * y^2 = x^3 + 3 or with a coordinate >= q, sets verdict_i = reject; the party still finishes.  So any deviation gives
 * B200_ERR_MAC on every honest party, and the outputs (proof, challenges, link shares, eta) are written only after the
 * check passed.  B200_ERR_UNSATISFIED is returned only after the check passed (an unsatisfied witness skips to it).
 * Security with abort: a deviating party can make the call fail but not make it succeed with a wrong result, except
 * with probability about (log length + 2) / r per call.
 *
 * Messages, against the plain call: exchange 0 carries H(seed_i) (32 bytes) after the 64-byte statement in a proof, and
 * after the partial quotient commitment in a link; then three more exchanges, each with the 32-byte header:
 *   seed reveal:   seed_i (32 bytes)
 *   check commit:  keccak256(record_i) (32 bytes)
 *   check reveal:  record_i = sigma_i (32) || Sigma_pt,i (64, affine, the identity as zeros) || verdict_i (32: byte 0 is
 *                  1 for accept, the rest zero) || salt_i (32)  (160 bytes)
 * H is keccak256.  A proof whose degree check fails skips rounds 4-5, a link whose exactness check fails skips the
 * opening; both go straight to these exchanges. */
/* Preprocessing with MACs (the counts of b200_mpc_prep_size): a_mac, b_mac, c_mac, masks_mac are this party's MAC shares
 * of the triples and masks.  Only b200_mpc_prove_auth accepts it; single use. */
int b200_mpc_prep_load_auth(b200_ctx* ctx, const b200_pk* pk, const uint64_t* a, const uint64_t* b, const uint64_t* c,
                            const uint64_t* a_mac, const uint64_t* b_mac, const uint64_t* c_mac, const uint64_t* masks,
                            const uint64_t* masks_mac, b200_mpc_prep** out);
/* INSECURE, as b200_mpc_prep_dealer (the same triples and masks for the same seed): alpha and every MAC share are derived
 * from the seed on the device; mac_key_share receives this party's alpha_i. */
int b200_mpc_prep_dealer_auth(b200_ctx* ctx, const b200_pk* pk, uint64_t seed, int party, int parties,
                              uint64_t mac_key_share[4], b200_mpc_prep** out);
/* INSECURE input stand-in for tests and benchmarks: this party's authenticated shares (shares, macs: count x 4 limbs each)
 * of `count` values the caller knows in full, under the MAC key b200_mpc_prep_dealer_auth derives from the same seed.
 * The share masks depend only on (seed, index): two tables shared under one seed get the same masks.  In production
 * the input protocol of the MPC framework produces these. */
int b200_mpc_dealer_share_auth(b200_ctx* ctx, uint64_t seed, int party, int parties, const uint64_t* values, size_t count,
                               uint64_t* shares, uint64_t* macs);
/* b200_mpc_prove on authenticated shares: wire_macs (5 x n) and blinder_macs (17) are the MAC shares of wire_shares and
 * blinder_shares; link_poly_mac (n + 2, may be NULL) receives the MAC shares of the linking polynomial.  The opened proof
 * equals b200_plonk_prove on the summed wires and blinders.  B200_ERR_INVALID for a preprocessing without MACs. */
int b200_mpc_prove_auth(b200_ctx* ctx, const b200_pk* pk, const b200_mpc_transport* transport, b200_mpc_prep* prep,
                        const uint64_t* mac_key_share, const uint64_t* wire_shares, const uint64_t* wire_macs,
                        const uint64_t* pub_inputs, const uint64_t* blinder_shares, const uint64_t* blinder_macs,
                        b200_proof* proof, uint64_t* link_poly_share, uint64_t* link_poly_mac, uint64_t* challenges);
/* b200_mpc_link on authenticated hints.  A plaintext hint (a validity proof's) is input by its holder through the MPC
 * framework's input protocol; "plaintext here, zeros elsewhere" has no valid MACs. */
int b200_mpc_link_auth(b200_ctx* ctx, const b200_bases* srs, const b200_mpc_transport* transport,
                       const uint64_t* mac_key_share, const uint64_t* a1_share, const uint64_t* a1_mac, size_t len1,
                       const uint64_t* a2_share, const uint64_t* a2_mac, size_t len2, const uint64_t* comm1,
                       const uint64_t* comm2, unsigned alignment, size_t offset, size_t size, b200_link_proof* proof,
                       uint64_t* eta);

/* ---- witness-side batch hashing (SURVEY.md §8(f) f4) ------------------------------------- */
/* `batch` independent Poseidon2 sponge hashes of `len` scalars each (inputs: batch x len x 4
 * limbs, Montgomery; out: batch x 4 limbs; host or device pointers).  Each equals the reference's
 * `compute_poseidon_hash(&values)` / `Poseidon2Sponge::new().hash(&values)`
 * (crates/crypto/src/hash/mod.rs:12-18, poseidon2.rs:38-44): t = 3, rate 2, R_F = 8, R_P = 56,
 * alpha = 5, constants of crates/crypto/src/hash/constants.rs. */
int b200_poseidon2_hash_batch(b200_ctx* ctx, const uint64_t* inputs, size_t batch, size_t len,
                              uint64_t* out);
/* `batch` bare permutations of 3-element states, in place (`Poseidon2Sponge::permute`,
 * poseidon2.rs:90-110). */
int b200_poseidon2_permute_batch(b200_ctx* ctx, uint64_t* states, size_t batch);

/* Roots of `batch` Merkle openings of `height` levels: leaf_hashes[i] is hashed up with its sister nodes
 * (sisters[i * height + lvl], bottom-up); is_right[i * height + lvl] != 0 means the running hash is the RIGHT child at
 * that level, i.e. the node is H(sister, cur), else H(cur, sister) — two-to-one Poseidon2 sponge hashes.  The native
 * side of `PoseidonMerkleHashGadget::compute_root` (circuits-core/src/zk_gadgets/primitives/merkle.rs:13-126) /
 * `MerkleOpening::compute_root`, for the batches witness generation walks (state_wrapper.rs:125-247). */
int b200_poseidon2_merkle_root_batch(b200_ctx* ctx, const uint64_t* leaf_hashes, const uint64_t* sisters,
                                     const uint8_t* is_right, size_t batch, unsigned height, uint64_t* roots);
/* `count` consecutive outputs of `batch` Poseidon CSPRNG streams (darkpool-types/src/csprng.rs:30-75: value i of a
 * stream is H(seed, i)): out[s * count + j] = H(seeds[s], first_index[s] + j).  The share / recovery streams behind
 * every `StateWrapper` (stream-cipher pads, recovery identifiers). */
int b200_poseidon2_csprng_batch(b200_ctx* ctx, const uint64_t* seeds, const uint64_t* first_index, size_t batch,
                                size_t count, uint64_t* out);

/* Keccak-256 of the transcript (host; exported so the hash can be pinned by known answers). */
void b200_keccak256(const uint8_t* data, size_t len, uint8_t out[32]);

/* ---- device self-test ------------------------------------------------------------------ */
/* Runs `iters` random Fr and Fq products through the production multiplier (IMAD.WIDE chains)
 * and the word-serial reference multiplier on the device and returns the number of
 * mismatches in *mismatches (0 expected). */
int b200_selftest_field(b200_ctx* ctx, uint64_t seed, size_t iters, uint64_t* mismatches);
/* out[i] = a[i] (op) b[i] on the device; field: 0 = Fr, 1 = Fq; op: 0 mul, 1 add, 2 sub,
 * 3 inverse of a.  Host buffers, n x 4 limbs (Montgomery).  For parity tests. */
int b200_field_op(b200_ctx* ctx, int field, int op, const uint64_t* a, const uint64_t* b, size_t n,
                  uint64_t* out);

#ifdef __cplusplus
}
#endif
#endif /* B200PROVER_H */
