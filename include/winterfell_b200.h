/* winterfell_b200.h — C ABI of the B200-native STARK proving hot path.
 *
 * Drop-in boundary for facebook/winterfell v0.13.1 (reference paths relative to /root/reference):
 * the library sits behind the four plug-in traits the reference's `Prover` selects through
 * associated types (prover/src/lib.rs:125-158): `TraceLde` (prover/src/trace/trace_lde/mod.rs:26-76),
 * `ConstraintEvaluator` (prover/src/constraints/evaluator/mod.rs:28-42), `ConstraintCommitment`
 * (prover/src/constraints/commitment/mod.rs:24-37) and `VectorCommitment`
 * (crypto/src/commitment.rs:28-86), plus the concrete FriProver (fri/src/prover/mod.rs:100-300)
 * that a GPU prover replaces by overriding `Prover::generate_proof` (prover/src/lib.rs:282).
 * INTEGRATION.md shows the Rust shim (`impl TraceLde for GpuTraceLde` ...) binding every entry
 * point below.
 *
 * Conventions
 *  - plain pointers and sizes only; every function returns WF_OK (0) or a negative error code and
 *    records a message retrievable with wf_last_error(). The Rust traits are infallible
 *    (they panic on misuse, e.g. trace_lde/default/mod.rs:150-158): the shim turns non-zero into panic!.
 *  - field elements are 64-bit words. `mont` flags say whether a HOST buffer holds the reference's
 *    in-memory Montgomery words (x * 2^64 mod p — what a Rust `&[BaseElement]` reinterpreted as
 *    `*const u64` exposes, math/src/field/f64/mod.rs:57-64,212-217) or canonical values in [0, p).
 *    Device buffers are always canonical. Digests are 32 bytes (Blake3_256 bytes, or the four
 *    canonical LE words of an Rp64_256 digest, rescue/rp64_256/digest.rs:36-45).
 *  - one wf_ctx per prover object / per GPU; calls on one ctx are issued on its CUDA stream in
 *    program order and are not re-entrant (the reference calls the factories sequentially from
 *    the proving thread, prover/src/lib.rs:282-492).
 *  - there is NO CPU fallback: every entry point fails with WF_ERR_CUDA when no sm_100 device is
 *    usable.
 */
#ifndef WINTERFELL_B200_H
#define WINTERFELL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WF_OK 0
#define WF_ERR_CUDA (-1)
#define WF_ERR_INVALID (-2)
#define WF_ERR_UNSUPPORTED (-3)
#define WF_ERR_STATE (-4)

#define WF_HASH_BLAKE3_256 0 /* crypto/src/hash/blake/mod.rs:21 */
#define WF_HASH_RP64_256 1   /* crypto/src/hash/rescue/rp64_256/mod.rs:118 */
#define WF_HASH_RPJIVE64_256 2 /* crypto/src/hash/rescue/rp64_256_jive/mod.rs:112 (Jive compression for merges) */
#define WF_HASH_SHA3_256 4     /* crypto/src/hash/sha/mod.rs:19 */
#define WF_HASH_BLAKE3_192 3   /* crypto/src/hash/blake/mod.rs:73: 24-byte digests. Digests cross this ABI in 32-byte slots (the last
                                * 8 bytes zero, as ByteDigest::as_bytes pads them); proofs carry 24 bytes per digest */

typedef struct wf_ctx wf_ctx;
typedef struct wf_mat wf_mat;   /* device matrix of base-field columns (segment layout, see DESIGN.md) */
typedef struct wf_tree wf_tree; /* device Merkle tree: leaves + nodes (crypto/src/merkle/mod.rs:86-98) */
typedef struct wf_fri wf_fri;   /* FRI prover state (fri/src/prover/mod.rs:100-116) */

/* ---- context ---------------------------------------------------------------------------------- */
/* `stream` is a cudaStream_t (NULL = legacy default stream). */
int wf_ctx_create(wf_ctx** out, int device, void* stream);
void wf_ctx_destroy(wf_ctx* ctx);
const char* wf_last_error(const wf_ctx* ctx);
/* One wf_ctx belongs to one device and one calling thread at a time; the library makes ctx's device current on the calling thread
 * wherever work for it starts (allocation, transform launch, gather, sync), so a process may hold contexts for several GPUs. */
int wf_ctx_sync(wf_ctx* ctx);
/* number of kernels this ctx has launched since creation (bench.py's gpu_launches) */
uint64_t wf_ctx_launch_count(const wf_ctx* ctx);
/* device memory this ctx holds: buffers handed out and not yet freed (count and bytes: the matrices, trees, FRI layers the
 * caller still owns) and bytes parked in the ctx's pool for reuse. After every handle is freed, live_buffers is 0 — also
 * after a call that returned an error. Any of the pointers may be NULL. */
int wf_ctx_mem_stats(const wf_ctx* ctx, uint64_t* live_buffers, uint64_t* live_bytes, uint64_t* pooled_bytes);
const char* wf_version(void);
/* stage tracing (the reference's `tracing` spans, prover/src/lib.rs:312-466): when on, the proving
 * entry points record a CUDA event at every stage boundary; wf_ctx_stage_times returns the stage
 * names (comma separated) and their durations in ms since the previous boundary, and resets. */
int wf_ctx_set_profiling(wf_ctx* ctx, int on);
int wf_ctx_stage_times(wf_ctx* ctx, char* names, size_t names_cap, float* ms, size_t* count);

/* ---- matrices --------------------------------------------------------------------------------- */
/* ColMatrix<E> (prover/src/matrix/col_matrix.rs:33): `ncols` host columns of `nrows` elements of
 * extension degree `ext_degree`; becomes ncols*ext_degree base columns on the device. The copies are enqueued on the ctx
 * stream: with PINNED host memory they are asynchronous, and the columns must stay valid and unmodified until the next call that
 * synchronises the context (wf_ctx_sync, any wf_*_root / *_to_host / wf_prove_*); pageable memory is staged before return. */
int wf_mat_from_host_columns(wf_ctx* ctx, const uint64_t* const* cols, uint32_t ncols, size_t nrows,
                             int ext_degree, int mont, wf_mat** out);
/* same, from a DEVICE buffer laid out column-major [ncols][nrows] (base columns, canonical) */
int wf_mat_from_device_columns(wf_ctx* ctx, const uint64_t* d_cols, uint32_t ncols, size_t nrows, wf_mat** out);
/* new matrix holding base columns [first, first + count) of m */
int wf_mat_select_columns(wf_ctx* ctx, const wf_mat* m, uint32_t first, uint32_t count, wf_mat** out);
int wf_mat_free(wf_ctx* ctx, wf_mat* m);
size_t wf_mat_rows(const wf_mat* m);
uint32_t wf_mat_cols(const wf_mat* m);
/* copy out as column-major [cols][rows] or row-major [rows][cols]; dst is host (to_host=1) or device */
int wf_mat_to_columns(wf_ctx* ctx, const wf_mat* m, uint64_t* dst, int to_host, int mont);
int wf_mat_to_rows(wf_ctx* ctx, const wf_mat* m, uint64_t* dst, int to_host, int mont);
/* rows at `positions` (k x cols words, canonical unless mont) -> host; TraceLde::query values
 * (trace_lde/default/mod.rs:199-230, build_segment_queries :284-297) */
int wf_mat_read_rows(wf_ctx* ctx, const wf_mat* m, const uint64_t* positions, size_t k, uint64_t* dst, int mont);

/* ColMatrix::interpolate_columns (col_matrix.rs:192-202): evaluations over the size-n subgroup
 * -> coefficients. n = rows must be a power of two >= 2. */
int wf_mat_interpolate(wf_ctx* ctx, const wf_mat* evals, wf_mat** polys);
/* fft::evaluate_poly per column (math/src/fft/mod.rs:85): coefficients -> evaluations, natural order */
int wf_mat_evaluate(wf_ctx* ctx, const wf_mat* polys, wf_mat** evals);
/* RowMatrix::evaluate_polys_over::<8> (row_matrix.rs:84-100): LDE over the coset 7 * <w_N>,
 * N = n << log_blowup, row i <-> point 7 * w_N^i (natural order). */
int wf_mat_lde(wf_ctx* ctx, const wf_mat* polys, uint32_t log_blowup, wf_mat** lde);
/* same, into a matrix the caller provides (e.g. a wf_mat_wrap_device view of a collective's send buffer) */
int wf_mat_lde_into(wf_ctx* ctx, const wf_mat* polys, uint32_t log_blowup, wf_mat* lde);
/* non-owning handle over device memory that already holds a rows x cols matrix in segment layout
 * (ceil(cols / W) segments of rows x W words, W = 8 for cols >= 8, else the next power of two >= cols);
 * wf_mat_free releases the handle, not the memory */
int wf_mat_wrap_device(wf_ctx* ctx, uint64_t* d_segments, size_t rows, uint32_t cols, wf_mat** out);
/* DefaultTraceLde::new up to the commitment (prover/src/trace/trace_lde/default/mod.rs:63-100,
 * build_trace_commitment :245-265) straight from HOST columns: equivalent to wf_mat_from_host_columns ->
 * wf_mat_interpolate -> wf_mat_lde, but the upload of column chunk k+1 overlaps the layout / iNTT / LDE of
 * chunk k (pass pinned host memory to get the overlap). Returns the coefficient matrix (TracePolyTable)
 * and the LDE. */
int wf_trace_lde_from_host(wf_ctx* ctx, const uint64_t* const* cols, uint32_t ncols, size_t nrows, int mont, uint32_t log_blowup,
                           wf_mat** polys, wf_mat** lde);
/* fft::interpolate_poly_with_offset per column (math/src/fft/mod.rs:351) */
int wf_mat_interpolate_with_offset(wf_ctx* ctx, const wf_mat* evals, uint64_t domain_offset, wf_mat** polys);

/* ---- commitments ------------------------------------------------------------------------------ */
/* RowMatrix::commit_to_rows (row_matrix.rs:184-228) with partition_size == num_cols, then
 * MerkleTree::new (crypto/src/merkle/mod.rs:116-135). */
int wf_commit_rows(wf_ctx* ctx, int hash_id, const wf_mat* m, wf_tree** out);
/* same with column partitions (row_matrix.rs:204-223): the row digest is H::merge_many of the digests of
 * chunks of `partition_size` BASE columns — partition_size = PartitionOptions::partition_size::<E>(cols)
 * * E::EXTENSION_DEGREE (air/src/options.rs:428-444); at most 16 partitions. 0 = whole rows. */
int wf_commit_rows_partitioned(wf_ctx* ctx, int hash_id, const wf_mat* m, uint32_t partition_size, wf_tree** out);
/* MerkleTree::new from host/device leaf digests (VectorCommitment::new, crypto/src/commitment.rs:41) */
int wf_tree_from_leaves(wf_ctx* ctx, int hash_id, const uint8_t* leaves, size_t nleaves, int leaves_on_device,
                        wf_tree** out);
int wf_tree_free(wf_ctx* ctx, wf_tree* t);
int wf_tree_root(wf_ctx* ctx, const wf_tree* t, uint8_t root[32]); /* VectorCommitment::commitment */
size_t wf_tree_num_leaves(const wf_tree* t);
/* copies leaves (nleaves*32 B) and nodes (nleaves*32 B) to host: MerkleTree::from_raw_parts inputs
 * (crypto/src/merkle/mod.rs:148) */
int wf_tree_to_host(wf_ctx* ctx, const wf_tree* t, uint8_t* leaves, uint8_t* nodes);
/* VectorCommitment::open_many = MerkleTree::prove_batch (merkle/mod.rs:217-272): writes the k leaf
 * digests (in the order of `positions`) and the serialized BatchMerkleProof (proofs.rs:390-401).
 * *proof_len: in = capacity, out = bytes written. */
int wf_tree_open_many(wf_ctx* ctx, const wf_tree* t, const uint64_t* positions, size_t k, uint8_t* leaves_out,
                      uint8_t* proof, size_t* proof_len);

/* ---- FRI (fri/src/prover/mod.rs) --------------------------------------------------------------- */
/* FriProver::new + build_layers (:179-239) over `len` evaluations of extension degree d held in
 * device matrix `evals` (d base columns, len rows), domain offset 7.
 * The transcript is the caller's: after each layer the library calls `commit(user, root32)` and
 * then `draw_alpha(user, alpha_out[d])` (ProverChannel::commit_fri_layer / draw_fri_alpha,
 * fri/src/prover/channel.rs:20-27); after the remainder it calls commit(user, remainder_hash). */
typedef void (*wf_fri_commit_fn)(void* user, const uint8_t root[32]);
typedef void (*wf_fri_draw_fn)(void* user, uint64_t* alpha_out);
int wf_fri_build_layers(wf_ctx* ctx, int hash_id, const wf_mat* evals, int ext_degree, uint32_t folding_factor,
                        uint32_t remainder_max_degree, uint32_t blowup, wf_fri_commit_fn commit,
                        wf_fri_draw_fn draw_alpha, void* user, wf_fri** out);
/* same, with the library's own DefaultProverChannel-style coin seeded with hash_elements([])
 * (fri/src/prover/channel.rs:60-72); roots_out receives (num_layers + 1) x 32 bytes. */
int wf_fri_build_layers_default_channel(wf_ctx* ctx, int hash_id, const wf_mat* evals, int ext_degree,
                                        uint32_t folding_factor, uint32_t remainder_max_degree, uint32_t blowup,
                                        uint8_t* roots_out, size_t roots_cap, wf_fri** out);
uint32_t wf_fri_num_layers(const wf_fri* f);
/* remainder polynomial, reversed coefficients (fri/src/prover/mod.rs:230-239); returns element count */
size_t wf_fri_remainder(const wf_fri* f, uint64_t* coeffs, size_t cap_words);
/* FriProver::build_proof (:254-296) serialized as FriProof (fri/src/proof.rs): *len in=cap, out=bytes */
int wf_fri_build_proof(wf_ctx* ctx, wf_fri* f, const uint64_t* positions, size_t k, uint8_t* out, size_t* len);
int wf_fri_free(wf_ctx* ctx, wf_fri* f);

/* ---- full proof (Prover::prove / generate_proof, prover/src/lib.rs:250-492) --------------------- */
/* Proves the built-in AIR family "FibSmall x k" (k copies of examples/src/fibonacci/fib_small/air.rs
 * side by side, trace width 2k; k = 1 is the reference's fib_small example) and writes the
 * serialized Proof (air/src/proof/mod.rs:189-200). trace_cols: 2k host columns of 2^log_n words;
 * results: the k public inputs (last value of column 2j+1).
 * opts[9] = { num_queries, blowup, grinding, field_extension (1|2|3), fri_folding, fri_remainder_max_degree,
 *             constraint batching (0 Linear | 1 Algebraic | 2 Horner), DEEP batching,
 *             hash_id | num_partitions << 8 | hash_rate << 16 }
 * (ProofOptions::new, air/src/options.rs:132; the two upper fields of opts[8] are ProofOptions::with_partitions,
 * options.rs:193-200 — 0 means the default PartitionOptions::new(1, 1); with more than one partition the main, auxiliary
 * and constraint commitments hash every row as merge_many of the digests of its column partitions, row_matrix.rs:204-223,
 * and the two bytes are written into the proof's serialized options). *proof_len: in = capacity, out = bytes written. */
int wf_prove_fib(wf_ctx* ctx, const uint64_t* const* trace_cols, int mont, uint32_t k, uint32_t log_n,
                 const uint64_t* results, const uint32_t* opts, uint8_t* proof, size_t* proof_len);

/* Generic single-segment AIR: Air::evaluate_transition (air/src/air/mod.rs:210) described as a
 * straight-line program, so that user AIRs beyond the built-in family run on the device evaluator.
 * air_desc (u64 words):
 *   [width, nT, {base_degree, ncycles, cycle...} x nT        TransitionConstraintDegree (transition/degree.rs)
 *    nP, {len, values...} x nP                               get_periodic_column_values (air/mod.rs:300)
 *    nC, constants...,  num_regs,  nI, {op, dst, a, b} x nI   registers: [0,w) current row, [w,2w) next row,
 *                                                             [2w,2w+nP) periodic values, then temporaries;
 *                                                             op 0 ADD, 1 SUB, 2 MUL (dst = r[a] op r[b]),
 *                                                             3 CONST (dst = constants[a]), 4 OUT (result[dst] = r[a])
 *    nA, {column, first_step, stride, nvals, values...} x nA  Assertion::single (stride 0, 1 value) / ::periodic
 *                                                             (stride > 0, 1 value) / ::sequence (stride > 0,
 *                                                             nvals = n / stride values) (assertions/mod.rs:62-120)
 *    nPub, public input elements...,  num_transition_exemptions]
 * Multi-segment descriptions go through wf_prove_air_aux. */
int wf_prove_air(wf_ctx* ctx, const uint64_t* air_desc, size_t air_desc_len, const uint64_t* const* trace_cols, int mont,
                 uint32_t log_n, const uint32_t* opts, uint8_t* proof, size_t* proof_len);

/* Multi-segment AIR (one auxiliary segment, as in the reference: air/src/air/trace_info.rs:24-40).
 * The description above is followed by the aux section
 *   [aux_width, num_rand_elements,
 *    nTa, {base_degree, ncycles, cycle...} x nTa            aux_transition_constraint_degrees (context.rs:93)
 *    aux_num_regs, nIa, {op, dst, a, b} x nIa                Air::evaluate_aux_transition (air/mod.rs:248-260):
 *                                                            registers over E: [0,w) main current, [w,2w) main next,
 *                                                            [2w,2w+aw) aux current, [2w+aw,2w+2aw) aux next, then
 *                                                            nP periodic values, then the random elements, then
 *                                                            temporaries; same opcodes
 *    nAa, {column, first_step, stride, nvals, {v0, v1, v2} x nvals} x nAa]   Air::get_aux_assertions (:279),
 *                                                            values in E (first ext words used)
 * After the main commitment the prover draws num_rand_elements E elements from the public coin
 * (Air::get_aux_rand_elements, air/mod.rs:292-306) and calls `aux_builder` (Prover::build_aux_trace,
 * prover/src/lib.rs:236-247) on the HOST: rand_elements = [num_rand][d] words, aux_out = [aux_width][n][d]
 * words (one Vec<E> per column, as ColMatrix<E>), both in the representation selected by `mont`.
 * The builder returns 0 on success. d = opts.field_extension. */
typedef int (*wf_aux_builder_fn)(void* user, const uint64_t* rand_elements, uint64_t* aux_out);
int wf_prove_air_aux(wf_ctx* ctx, const uint64_t* air_desc, size_t air_desc_len, const uint64_t* const* trace_cols, int mont,
                     uint32_t log_n, const uint32_t* opts, wf_aux_builder_fn aux_builder, void* aux_user, uint8_t* proof,
                     size_t* proof_len);

/* Same, for AIRs whose auxiliary assertions depend on the random elements (Air::get_aux_assertions(&self, aux_rand_elements),
 * air/src/air/mod.rs:279): after the random elements are drawn — and after aux_builder has run — `aux_assertions` is called
 * on the HOST with the same rand_elements and with `values` = [sum of nvals over the aux assertions][d] words in description
 * order, preloaded with the description's values; what it leaves there is asserted (positions, strides and counts stay the
 * description's). Representation selected by `mont`; returns 0 on success. A verifier must apply the same function. */
typedef int (*wf_aux_assertions_fn)(void* user, const uint64_t* rand_elements, uint64_t* values);
int wf_prove_air_aux_dyn(wf_ctx* ctx, const uint64_t* air_desc, size_t air_desc_len, const uint64_t* const* trace_cols, int mont,
                         uint32_t log_n, const uint32_t* opts, wf_aux_builder_fn aux_builder, wf_aux_assertions_fn aux_assertions,
                         void* aux_user, uint8_t* proof, size_t* proof_len);

/* same, trace already on the device: column-major [2k][2^log_n], canonical words */
int wf_prove_fib_dev(wf_ctx* ctx, const uint64_t* d_trace, uint32_t k, uint32_t log_n, const uint64_t* results,
                     const uint32_t* opts, uint8_t* proof, size_t* proof_len);

/* ---- the same pipeline as separate steps, for a host that owns the transcript (the Rust shim of
 *      INTEGRATION.md: impl ConstraintEvaluator / ConstraintCommitment, prover/src/lib.rs:195-223) ---- */
/* ConstraintEvaluator::evaluate (prover/src/constraints/evaluator/mod.rs:28-42, default.rs:60-118) +
 * ConstraintEvaluationTable::combine (evaluation_table.rs:163): CompositionPolyTrace over the CE domain
 * as a (n * ce_blowup) x ext matrix. air_desc as for wf_prove_air[_aux]; main_lde N x width, aux_lde
 * N x aux_width*ext (NULL for single-segment AIRs). coeffs: ConstraintCompositionCoefficients
 * (air/src/air/coefficients.rs:72) flattened [transition: main, aux | boundary: main, aux][ext] with
 * boundary coefficients in the sorted-assertion order; aux_rand [num_rand][ext]. Canonical words. */
int wf_eval_constraints(wf_ctx* ctx, const uint64_t* air_desc, size_t air_desc_len, uint32_t log_n, uint32_t blowup, uint32_t ext,
                        const wf_mat* main_lde, const wf_mat* aux_lde, const uint64_t* coeffs, const uint64_t* aux_rand,
                        wf_mat** out);
/* Prover::build_constraint_commitment (prover/src/lib.rs:215-223; DefaultConstraintCommitment::new,
 * constraints/commitment/default.rs:44-150): composition trace -> num_cols column polynomials of
 * degree < n (CompositionPoly, n x num_cols*ext), their LDE (N x num_cols*ext) and its row commitment */
int wf_composition_commit(wf_ctx* ctx, int hash_id, const wf_mat* comp_trace, uint32_t log_n, uint32_t blowup, uint32_t ext,
                          uint32_t num_cols, wf_mat** polys, wf_mat** lde, wf_tree** tree);
/* same with the PartitionOptions argument of build_constraint_commitment (lib.rs:220): partition_size in BASE columns =
 * PartitionOptions::partition_size::<E>(num_cols) * ext (0 or num_cols * ext = whole rows), as wf_commit_rows_partitioned */
int wf_composition_commit_partitioned(wf_ctx* ctx, int hash_id, const wf_mat* comp_trace, uint32_t log_n, uint32_t blowup,
                                      uint32_t ext, uint32_t num_cols, uint32_t partition_size, wf_mat** polys, wf_mat** lde,
                                      wf_tree** tree);
/* ColMatrix::evaluate_columns_at (prover/src/matrix/col_matrix.rs:245) at two points of E (z and z*g for
 * TracePolyTable::get_ood_frame, trace/poly_table.rs:68-76; CompositionPoly::get_ood_frame,
 * composition_poly.rs:101-108). col_ext = 1: base columns; col_ext = ext: the matrix holds columns of E
 * (ext consecutive base columns each). out0/out1: [cols / col_ext][ext] host words. */
int wf_mat_evaluate_at(wf_ctx* ctx, const wf_mat* polys, uint32_t ext, uint32_t col_ext, const uint64_t* z0, const uint64_t* z1,
                       uint64_t* out0, uint64_t* out1);
/* DeepCompositionPoly::{add_trace_polys, add_composition_poly, evaluate} (prover/src/composer/mod.rs:67-210):
 * DEEP composition evaluated over the LDE domain, N x ext. coeffs / ood_cur / ood_next: [width + aux_width +
 * composition columns][ext] in that order (DeepCompositionCoefficients, TraceOodFrame + QuotientOodFrame rows). */
int wf_deep_compose(wf_ctx* ctx, uint32_t ext, const wf_mat* main_lde, const wf_mat* aux_lde, const wf_mat* cons_lde, uint32_t log_n,
                    const uint64_t* z, const uint64_t* coeffs, const uint64_t* ood_cur, const uint64_t* ood_next, wf_mat** out);

/* ProverChannel::grind_query_seed (prover/src/channel.rs:169-184), serial semantics: the SMALLEST
 * nonce >= 1 with trailing_zeros(first 8 LE bytes of H::merge_with_int(seed, nonce)) >= grinding. */
int wf_grind(wf_ctx* ctx, int hash_id, const uint8_t seed[32], uint32_t grinding, uint64_t* nonce);

/* ---- one proof sharded over several GPUs (SURVEY.md 8e; one process and one wf_ctx per GPU) ------------------
 * The reference has no distributed prover; its unit of distribution is the column (ColMatrix columns are independent,
 * prover/src/matrix/col_matrix.rs:192-202) and PartitionOptions (air/src/options.rs:405-445). Here rank r of `world`
 * owns a block of whole 8-column segments of the trace (wf_host_shard_columns): it interpolates and extends them locally, the LDE is exchanged into
 * row shards (rank r holds LDE rows [r*N/world, (r+1)*N/world) of ALL columns plus `blowup` halo rows), and leaf
 * hashing, constraint evaluation, DEEP composition and the first FRI layers run on row shards; every Merkle tree is a
 * local subtree per rank plus log2(world) top levels built from an all-gather of the subtree roots; query openings are
 * gathered from their owners. The proof is byte-identical to wf_prove_fib's on one GPU.
 * The host program supplies the collectives (NCCL point-to-point in bench.py; any MPI-like layer works): */
typedef struct wf_comm {
    void* user;
    int rank, world; /* world: a power of two */
    /* Point-to-point exchange of DEVICE buffers of `bytes` bytes each: send[i] goes to rank send_peer[i], recv[i] is
     * filled by rank recv_peer[i]; transfers between one pair of ranks match in list order; no entry names the caller's
     * own rank. Must be ordered after the work already enqueued on the ctx stream and be complete, or ordered on that
     * stream, when it returns. */
    int (*exchange)(void* user, size_t nsend, const int* send_peer, const void* const* send, size_t nrecv,
                    const int* recv_peer, void* const* recv, size_t bytes);
    /* all-gather of `bytes` bytes per rank between HOST buffers: recv = world x bytes in rank order */
    int (*all_gather_host)(void* user, const void* send, void* recv, size_t bytes);
    /* element-wise wrapping sum over the ranks of `words` 64-bit words of a DEVICE buffer, in place (merges gathers
     * whose entries are non-zero on exactly one rank); same ordering rule as exchange */
    int (*all_reduce_sum)(void* user, void* d_buf, size_t words);
    /* Optional (may be NULL: every exchange is then ordered on the ctx stream). fork: exchanges issued from now on run on the
     * communicator's own stream, ordered after everything enqueued on the ctx stream so far — the library keeps enqueuing
     * kernels on the ctx stream meanwhile (the LDE of the next coset overlaps the exchange of the previous one). fork may
     * be called repeatedly; each call adds "wait for the ctx stream's current tail" to the communicator stream. join: the
     * ctx stream waits for every exchange issued since the first fork; later exchanges are on the ctx stream again. */
    int (*fork)(void* user);
    int (*join)(void* user);
} wf_comm;
/* FibSmall x k (as wf_prove_fib) sharded over comm->world GPUs: this rank passes ITS 2k/world columns (host columns, or
 * d_local = device column-major [2k/world][2^log_n]); 2k/world must be a multiple of 8 (whole 8-column segments).
 * `results` and `opts` are the full proof's; every rank returns the same proof bytes.
 * stats (optional, 8 doubles): [0] bytes this rank sent through exchanges ordered on the ctx stream, [1] ms inside those,
 * [2] number of collectives, [3] ms inside all_gather_host + all_reduce_sum, [4] FRI layers folded on shards, [5] bytes sent
 * overlapped with compute (the trace LDE's cosets), [6] how those travelled: 2 = written by the last LDE pass itself into the
 * owners' row shards mapped through CUDA IPC (stores over NVLink; the default when the driver allows it and world <= 8),
 * 1 = peer copies (copy engines) into mapped staging buffers, 0 = comm->exchange between fork and join (WF_PEER_PUSH=0). */
int wf_prove_fib_sharded(wf_ctx* ctx, const wf_comm* comm, const uint64_t* const* local_cols, const uint64_t* d_local, int mont,
                         uint32_t k, uint32_t log_n, const uint64_t* results, const uint32_t* opts, uint8_t* proof,
                         size_t* proof_len, double* stats);
/* Which trace columns rank `rank` of `world` owns in a sharded proof: the S = ceil(width / 8) segments are split
 * as evenly as possible. Rank r owns segments [floor(r S / world), floor((r+1) S / world)), which gives columns
 * [*first, *first + *count); *count may be 0. When 8 * world divides the width, these are the blocks wf_prove_fib_sharded
 * takes. width 1..255, world a power of two >= 2, 0 <= rank < world; WF_OK or WF_ERR_INVALID. Host-only. */
int wf_host_shard_columns(uint32_t width, int world, int rank, uint32_t* first, uint32_t* count);
/* wf_prove_air (single-segment description) sharded over comm->world GPUs. This rank passes the columns
 * wf_host_shard_columns names: host columns, or d_local = device column-major [count][2^log_n]; a rank that owns no
 * column passes NULL for both (it still takes part in every collective). air_desc, log_n and opts are the whole proof's
 * and must be the same on every rank. Every rank returns the same bytes, equal to wf_prove_air's on one GPU.
 * Before any device work every rank checks its own arguments (description, no aux segment: WF_ERR_UNSUPPORTED; world a
 * power of two >= 2; columns passed iff some are owned; blowup >= the constraints' blowup; at least 64 * blowup LDE rows and
 * 64 constraint-evaluation rows per rank) and the ranks all-gather (status, hash of description, log_n, opts, world): if
 * any rank refused, every rank returns the lowest refusing rank's status; if the hashes differ, every rank returns
 * WF_ERR_INVALID. No rank then waits on another. stats: as wf_prove_fib_sharded; [6] = 2 only when every rank owns the
 * same number of whole 8-column segments (the fused form needs it; other splits take the peer copies). */
int wf_prove_air_sharded(wf_ctx* ctx, const wf_comm* comm, const uint64_t* air_desc, size_t air_desc_len,
                         const uint64_t* const* local_cols, const uint64_t* d_local, int mont, uint32_t log_n,
                         const uint32_t* opts, uint8_t* proof, size_t* proof_len, double* stats);
/* Aux columns this rank builds: E columns [first_col, first_col + num_cols) of the aux segment, written to
 * aux_out = [num_cols][n][d] words (one Vec<E> per column, as wf_aux_builder_fn). Returns 0 on success. */
typedef int (*wf_aux_shard_builder_fn)(void* user, const uint64_t* rand_elements, uint32_t first_col, uint32_t num_cols,
                                       uint64_t* aux_out);
/* wf_prove_air_aux / wf_prove_air_aux_dyn (description WITH an aux segment) sharded over comm->world GPUs; every rank returns
 * the same bytes, equal to those one-GPU calls' for the same description, trace, builder and options. The main trace is
 * passed as in wf_prove_air_sharded.
 * Aux ownership: the aux segment is aw * d BASE columns (component q of E column j is base column j d + q) and rank r owns
 * base columns [first, first + count) = wf_host_shard_columns(aw * d, world, r). After the main commitment every rank draws
 * the same random elements (Montgomery form under `mont`, as wf_prove_air_aux) and calls aux_builder ONCE with the E columns
 * covering its base columns: first_col = first / d, num_cols = ceil((first + count) / d) - first_col; a rank that owns no aux
 * base column is not called. With d > 1 one E column can straddle two ranks: both build it and each keeps its own
 * components, so the builder must be deterministic. aux_assertions (NULL: the description's static aux assertions) is
 * called on EVERY rank as in wf_prove_air_aux_dyn; it must return the same values everywhere (Air::get_aux_assertions
 * depends only on public inputs and random elements).
 * Agreement: before any device work as wf_prove_air_sharded, plus WF_ERR_INVALID for a description without an aux segment,
 * a NULL aux_builder, or aux assertions that do not validate. After the callbacks the ranks all-gather (callback status,
 * hash of the aux assertion values): if a callback failed on any rank, every rank returns the lowest failing rank's status;
 * if the values differ, every rank returns WF_ERR_INVALID. stats: as wf_prove_air_sharded ([6] describes the main trace's
 * transport), and [7] = milliseconds this rank spent inside aux_builder and aux_assertions. */
int wf_prove_air_aux_sharded(wf_ctx* ctx, const wf_comm* comm, const uint64_t* air_desc, size_t air_desc_len,
                             const uint64_t* const* local_cols, const uint64_t* d_local, int mont, uint32_t log_n,
                             const uint32_t* opts, wf_aux_shard_builder_fn aux_builder,
                             wf_aux_assertions_fn aux_assertions /* NULL: static aux assertions */, void* aux_user,
                             uint8_t* proof, size_t* proof_len, double* stats);

/* ---- constraint kernels compiled per AIR ---------------------------------------------------------------------------
 * wf_eval_constraints / wf_prove_air[_aux] evaluate the AIR's transition programs with a kernel compiled at run time for that
 * AIR (NVRTC: the programs become straight-line code, registers and constants are literals), cached in the context; without
 * NVRTC on the machine, or with wf_ctx_set_jit(ctx, 0), the same programs are interpreted by the built-in kernel (same
 * results bit for bit). wf_ctx_jit_stats: kernels compiled, launches served from the cache, compilations that failed and
 * fell back. wf_jit_compile_air compiles the kernel of a description without a device (log: compiler output). */
int wf_ctx_set_jit(wf_ctx* ctx, int on);
int wf_ctx_jit_stats(wf_ctx* ctx, uint64_t* compiled, uint64_t* cache_hits, uint64_t* fallbacks);
int wf_jit_compile_air(const uint64_t* air_desc, size_t air_desc_len, uint32_t ext, size_t* cubin_bytes, char* log, size_t log_cap);
/* Everything wf_prove_air / wf_eval_constraints check about a description before they touch the device, without a device:
 * structure, degrees against the blowup factor, periodic columns, assertion validity and overlaps (the conditions
 * Air::new, BoundaryConstraints::new and prepare_assertions panic on, air/src/air/boundary/mod.rs:190-215). WF_OK, or
 * WF_ERR_INVALID with the reason in msg. */
int wf_air_check(const uint64_t* air_desc, size_t air_desc_len, uint32_t log_n, uint32_t blowup, char* msg, size_t msg_cap);

/* ---- plain kernels on caller-owned DEVICE buffers (unit parity + bench legs) ------------------- */
/* in-place NTT (inverse=0) / iNTT (inverse=1) of `cols` columns, column-major [cols][n], n = 1 << log_n */
int wf_ntt_dev(wf_ctx* ctx, uint64_t* d_data, uint32_t log_n, uint32_t cols, int inverse);
/* leaf digests of a row-major [nrows][cols] device matrix */
int wf_hash_rows_dev(wf_ctx* ctx, int hash_id, const uint64_t* d_rows, size_t nrows, uint32_t cols, uint8_t* d_digests);
/* Merkle nodes (nleaves x 32 B, nodes[0] = 0, nodes[1] = root) from device leaf digests */
int wf_merkle_dev(wf_ctx* ctx, int hash_id, const uint8_t* d_leaves, size_t nleaves, uint8_t* d_nodes);
/* one FRI fold: d_evals [len][d] -> d_next [len/folding][d]; alpha = d host words */
int wf_fri_fold_dev(wf_ctx* ctx, const uint64_t* d_evals, size_t len, int ext_degree, uint32_t folding_factor,
                    const uint64_t* alpha, uint64_t* d_next);

/* field arithmetic of the device code on caller-chosen operands (a, b: n canonical words each, device):
 * d_out[0..n) = a*b (math/src/field/f64/mod.rs:357), [n..2n) = a+b (:319), [2n..3n) = a-b (:339),
 * [3n..4n) = 1/a (:157; 0 for a = 0), then 18 blocks a * 2^s for s in WF_FIELD_TEST_SHIFTS.
 * d_out holds 22 n words. */
#define WF_FIELD_TEST_SHIFTS {1, 3, 6, 12, 24, 31, 32, 33, 48, 63, 64, 65, 72, 80, 84, 90, 95, 96}
int wf_field_ops_dev(wf_ctx* ctx, const uint64_t* d_a, const uint64_t* d_b, size_t n, uint64_t* d_out);
/* extension-field arithmetic of the device code (ExtensibleField<2> / <3> for BaseElement, math/src/field/f64/mod.rs:401-499;
 * inverses extensions/quadratic.rs:81-94, cubic.rs:81-97): a, b = n elements of `ext` (2 | 3) canonical words each (device);
 * d_out = 6 blocks of n elements: a*b, 1/a (0 for 0), frobenius(a), a.mul_base(b[0]), a+b, a-b. */
int wf_ext_ops_dev(wf_ctx* ctx, uint32_t ext, const uint64_t* d_a, const uint64_t* d_b, size_t n, uint64_t* d_out);

/* ---- host-side helpers of the product (transcript arithmetic; no GPU needed) ------------------- */
/* H::hash_elements / merge / merge_with_int on the host (crypto/src/hash/mod.rs:31-64) */
int wf_host_hash_elements(int hash_id, const uint64_t* elems, size_t n, uint8_t out[32]);
int wf_host_merge(int hash_id, const uint8_t two[64], uint8_t out[32]);
int wf_host_merge_with_int(int hash_id, const uint8_t seed[32], uint64_t value, uint8_t out[32]);
uint64_t wf_host_mul(uint64_t a, uint64_t b);           /* canonical Goldilocks product */
uint64_t wf_host_mul_2exp(uint64_t x, uint32_t k);      /* x * 2^k mod p, k <= 96 (kernel twiddle path) */
uint64_t wf_host_mont_to_canonical(uint64_t m);
uint64_t wf_host_canonical_to_mont(uint64_t x);
/* ByteWriter::write_usize (utils/core/src/serde/byte_writer.rs:77-92), the vint64 of the proof format;
 * returns the number of bytes written (1..9) */
size_t wf_host_write_usize(uint64_t value, uint8_t out[9]);
/* DefaultRandomCoin::new(seed elements) [+ reseed(digest)] + draw x count (crypto/src/random/default.rs:95-170):
 * the transcript arithmetic the proof path runs on the host. out[count][d]; 0 on success */
int wf_host_coin_draw(int hash_id, const uint64_t* seed_elems, size_t n_seed, const uint8_t* reseed32, int d, size_t count,
                      uint64_t* out);

/* index arithmetic of an opening in a tree stored as one subtree per rank (wf_prove_fib_sharded): want[i] = heap node
 * (< n_global) or n_global + leaf that MerkleTree::prove_batch (crypto/src/merkle/mod.rs:217-272) reads for `positions`;
 * idx[i] = its index in rank `rank`'s subtree (node < n_local, else n_local + leaf), ~0 when another rank holds it,
 * ~0 - 1 for a node of the top log2(world) levels. Returns the number of entries or -1. Host code. */
long wf_host_sharded_opening_plan(size_t n_global, int world, int rank, const uint64_t* positions, size_t k, uint64_t* want,
                                  uint64_t* idx, size_t cap);
/* FibSmallProver::build_trace (examples/src/fibonacci/fib_small/prover.rs:37-53) for the built-in "FibSmall x k"
 * family: cols = [2k][n] canonical words, pair j starting at (j+1, j+1); results[j] = its public input. Host code. */
int wf_host_build_fib_trace(uint32_t k, size_t n, uint64_t* cols, uint64_t* results);

#ifdef __cplusplus
}
#endif
#endif /* WINTERFELL_B200_H */
