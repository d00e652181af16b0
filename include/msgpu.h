/* libmsgpu -- C ABI of the B200 (sm_100a) commitment hot path for multi-stark.
 *
 * These are the entry points a Rust `msgpu-sys` crate binds (INTEGRATION.md shows the `extern "C"`
 * block and the `GpuDft` / `GpuFriPcs` wrappers that slot into `GoldilocksBlake3Config`,
 * reference src/types.rs:85,200,209-223). Conventions:
 *   - every function returns 0 on success and a negative code on failure; msgpu_last_error() gives the
 *     message of the last failure on the calling thread. Nothing aborts or throws across the ABI.
 *   - matrices are row-major arrays of canonical Goldilocks values (uint64_t < 2^64 - 2^32 + 1),
 *     i.e. the memory of a p3 `RowMajorMatrix<Goldilocks>` (reference src/prover.rs:336-351).
 *   - extension-field values (`BinomialExtensionField<Goldilocks, 2>`, X^2 = 7) are two adjacent
 *     uint64_t (c0, c1), the layout `flatten_to_base` produces (reference src/prover.rs:494-495).
 *   - a context owns one CUDA stream; calls on one context must come from one thread at a time
 *     (Send, not Sync -- the reference calls `prove` from a single thread, src/prover.rs:289).
 *   - host-pointer entry points copy their inputs to the device before returning and block until
 *     their outputs are written; `_dev` entry points take device pointers and are stream-ordered.
 */
#ifndef MSGPU_H
#define MSGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct msgpu_ctx msgpu_ctx;
/* Device-resident `Pcs::ProverData` / `Mmcs::ProverData`: the committed (LDE) matrices in
 * bit-reversed row order plus every digest layer of the Merkle tree. */
typedef struct msgpu_pdata msgpu_pdata;

#define MSGPU_OK 0
#define MSGPU_ERR_INVALID (-1) /* bad argument (the reference panics/asserts on these) */
#define MSGPU_ERR_CUDA (-2)    /* CUDA runtime failure; there is no CPU fallback */
#define MSGPU_ERR_INTERNAL (-3)

/* ---- context ---------------------------------------------------------------------------------- */
/* `stream`: a cudaStream_t to launch on (e.g. the caller's current stream) or NULL to create one. */
int msgpu_ctx_create(int device, void* stream, msgpu_ctx** out);
void msgpu_ctx_destroy(msgpu_ctx* ctx);
const char* msgpu_last_error(void);
int msgpu_sync(msgpu_ctx* ctx);
void* msgpu_stream(msgpu_ctx* ctx);
/* number of kernels this library has launched on the context (bench.py `gpu_launches`) */
uint64_t msgpu_launch_count(msgpu_ctx* ctx);

/* Per-launch timing with CUDA events on the context's stream (bench.py roofline). Between begin and
 * end every kernel launch of the library is bracketed by two events; end synchronises and writes a
 * JSON array [{"stage", "kernel", "launches", "ms"}] (NUL-terminated) into json_out. */
int msgpu_profile_begin(msgpu_ctx* ctx);
int msgpu_profile_end(msgpu_ctx* ctx, char* json_out, size_t cap);

/* ---- memory ----------------------------------------------------------------------------------- */
int msgpu_malloc(msgpu_ctx* ctx, size_t bytes, void** dptr);
int msgpu_free(msgpu_ctx* ctx, void* dptr);
int msgpu_memcpy_h2d(msgpu_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes);
int msgpu_memcpy_d2h(msgpu_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes);
int msgpu_host_alloc(size_t bytes, void** hptr); /* pinned host memory */
int msgpu_host_free(void* hptr);
/* Page-lock host memory the caller owns (the Vec behind a p3 `RowMajorMatrix<Goldilocks>`), so that the host-pointer entry points
 * read it directly over PCIe with no staging copy; unregister before the memory is freed. */
int msgpu_host_register(void* hptr, size_t bytes);
int msgpu_host_unregister(void* hptr);
/* Context options. MSGPU_OPT_CANONICALIZE_INPUTS = 1: host matrices handed to msgpu_commit / msgpu_upload_begin /
 * msgpu_upload_canonical may hold ANY u64 representative (p3's `Goldilocks` is `repr(transparent)` over a u64 that is not kept
 * reduced): they are reduced mod p on the device right after the upload instead of being rejected. Together with
 * msgpu_host_register this makes the reference's matrices uploadable with zero host-side copies. */
#define MSGPU_OPT_CANONICALIZE_INPUTS 1
int msgpu_ctx_set_option(msgpu_ctx* ctx, int option, uint64_t value);
/* H2D copy of n field elements that also verifies the ABI's precondition on the device: every value must be
 * canonical (< p). Returns MSGPU_ERR_INVALID otherwise (a typed `Goldilocks` can never be out of range in the
 * reference; raw u64 buffers can). */
int msgpu_upload_canonical(msgpu_ctx* ctx, void* dst_dev, const uint64_t* src_host, uint64_t n);

/* ---- TwoAdicSubgroupDft slot (reference: `type Dft = Radix2DitParallel<Val>`, src/types.rs:200;
 *      used at src/prover.rs:440,650,716) ------------------------------------------------------- */
/* dft_batch(m): out[k] = sum_j in[j] w^{jk}, natural order (rows x cols in, rows x cols out). */
int msgpu_dft_batch(msgpu_ctx* ctx, const uint64_t* in, uint64_t rows, uint64_t cols, uint64_t* out);
/* dft_batch(m).bit_reverse_rows(): the raw storage, natural index k at row rev(k)
 * (src/prover.rs:648-650,716). */
int msgpu_dft_batch_bitrev(msgpu_ctx* ctx, const uint64_t* in, uint64_t rows, uint64_t cols, uint64_t* out);
/* idft_batch(m): inverse of dft_batch, natural order. */
int msgpu_idft_batch(msgpu_ctx* ctx, const uint64_t* in, uint64_t rows, uint64_t cols, uint64_t* out);
/* coset_lde_batch(m, added_bits, shift).bit_reverse_rows(): what `Pcs::commit` stores per matrix,
 * out[i] = P(shift * w_{rows<<added_bits}^{rev(i)}) (src/prover.rs:681-692). */
int msgpu_coset_lde_batch_bitrev(msgpu_ctx* ctx, const uint64_t* in, uint64_t rows, uint64_t cols, uint32_t added_bits,
                                 uint64_t shift, uint64_t* out);
/* `lde_from_shifted_coefficients` (src/prover.rs:709-717): zero-pad to rows << added_bits, one DFT,
 * bit-reversed storage. */
int msgpu_lde_from_shifted_coefficients(msgpu_ctx* ctx, const uint64_t* in, uint64_t rows, uint64_t cols,
                                        uint32_t added_bits, uint64_t* out);
/* device-pointer forms (in and out are device buffers; out may not alias in) */
int msgpu_dft_batch_bitrev_dev(msgpu_ctx* ctx, const uint64_t* in, uint64_t rows, uint64_t cols, uint64_t* out);
int msgpu_coset_lde_batch_bitrev_dev(msgpu_ctx* ctx, const uint64_t* in, uint64_t rows, uint64_t cols,
                                     uint32_t added_bits, uint64_t shift, uint64_t* out);
int msgpu_lde_from_shifted_coefficients_dev(msgpu_ctx* ctx, const uint64_t* in, uint64_t rows, uint64_t cols,
                                            uint32_t added_bits, uint64_t* out);

/* ---- Pcs / Mmcs slot (reference: `type Pcs = TwoAdicFriPcs<Val, Dft, Mmcs, ExtMmcs>`,
 *      `type Mmcs = MerkleTreeMmcs<..Blake3..>`, src/types.rs:82-85,199-223) ---------------------- */
/* Pcs::commit (src/prover.rs:350,419; src/system.rs:193): per matrix the coset LDE with shift
 * GENERATOR = 7 in bit-reversed row order, then one MMCS over all LDEs. `mats[i]` is a HOST pointer
 * to heights[i] x widths[i] evaluations over the natural domain. root32 receives the 32-byte root
 * (cap_height 0). */
int msgpu_commit(msgpu_ctx* ctx, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths,
                 uint64_t n_mats, uint32_t log_blowup, msgpu_pdata** out, uint8_t* root32);
/* The same in two steps with the uploads on the context's COPY stream, so that matrix i is extended while matrices
 * i + 1 ... are still crossing PCIe (and anything enqueued on the copy stream in between, e.g. msgpu_claims_prefetch, travels
 * under the kernels). upload_begin returns at once; the host matrices (pinned memory for a real overlap) must stay valid until
 * commit_upload returns. commit_upload consumes the handle; verify_canonical = 1 checks every value < p on the device;
 * kept_inputs (optional, n_mats pointers out) receives the natural-order device copies, owned by the caller (msgpu_free);
 * local_only = 1 builds the local part of a sharded commitment (as msgpu_commit_local_dev: no tree, root32 may be NULL). */
typedef struct msgpu_upload msgpu_upload;
int msgpu_upload_begin(msgpu_ctx* ctx, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths,
                       uint64_t n_mats, msgpu_upload** out);
int msgpu_commit_upload(msgpu_upload* up, uint32_t log_blowup, int verify_canonical, uint64_t** kept_inputs, int local_only,
                        msgpu_pdata** out, uint8_t* root32);
void msgpu_upload_free(msgpu_upload* up);
/* same with DEVICE input pointers (inputs are not modified) */
int msgpu_commit_dev(msgpu_ctx* ctx, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths,
                     uint64_t n_mats, uint32_t log_blowup, msgpu_pdata** out, uint8_t* root32);
/* Pcs::commit_ldes (src/prover.rs:526): Merkle-only commitment to LDEs that already live on the
 * device in bit-reversed row order. The prover data BORROWS (take_ownership = 0) or adopts
 * (take_ownership = 1; buffers must come from msgpu_malloc) the matrices. */
/* root32 == NULL: nothing is read back and nothing waits (the root is the last digest of msgpu_pdata_digests). */
int msgpu_commit_ldes_dev(msgpu_ctx* ctx, uint64_t* const* ldes, const uint64_t* heights, const uint64_t* widths,
                          uint64_t n_mats, int take_ownership, msgpu_pdata** out, uint8_t* root32);
/* The same where some LDEs still exist as COLUMN BLOCKS (block_ptrs / block_widths[i * n_blocks + b]: dense heights[i] x width_b,
 * column order; a null first pointer = matrix i is already in ldes[i]): the leaf-hash pass reads the blocks -- which may live in
 * other GPUs' memory, msgpu_peers_ptr -- and writes the row-major matrix to ldes[i] as it hashes (fused gather + commit). */
int msgpu_commit_ldes_blocks_dev(msgpu_ctx* ctx, uint64_t* const* ldes, const uint64_t* heights, const uint64_t* widths, uint64_t n_mats,
                                 uint64_t n_blocks, const uint64_t* const* block_ptrs, const uint64_t* block_widths, int take_ownership,
                                 msgpu_pdata** out, uint8_t* root32);
/* ---- one commitment whose matrices live on several GPUs (SURVEY 8e, partitioning A: circuits -> GPUs) ----
 * The MMCS hashes, per LDE height, the rows of all matrices of that height into one leaf digest and injects the shorter
 * classes on the way up (p3-merkle-tree, src/types.rs:82-84). When every height class lives on ONE rank, a rank can hash
 * its classes alone (msgpu_commit_local_dev) and only the 32-byte-per-row class digests travel to the rank that builds
 * the node layers (msgpu_tree_from_digests); the root and all openings are then bit-identical to a single-GPU commit.
 * commit_local: `mats` are DEVICE pointers to this rank's matrices in commit order: evaluations (inputs_are_ldes = 0,
 * not modified) or finished LDEs from msgpu_malloc that the prover data adopts (inputs_are_ldes = 1). The result has no
 * tree: it serves msgpu_quotient, msgpu_open_begin and the ROW part of msgpu_open_batch_multi (0 sibling digests). */
int msgpu_commit_local_dev(msgpu_ctx* ctx, uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths,
                           uint64_t n_mats, uint32_t log_blowup, int inputs_are_ldes, msgpu_pdata** out);
uint64_t msgpu_pdata_num_classes(const msgpu_pdata* pd);
/* height class k (tallest first) of a local part: its LDE height and the device pointer of its 32 * height digest bytes */
int msgpu_pdata_class_digests(const msgpu_pdata* pd, uint64_t k, uint64_t* lde_height, uint8_t** dev_ptr);
/* node layers over the class digests of ALL ranks (device pointers, distinct power-of-two heights, any order; not
 * modified). The result has no matrices: msgpu_open_batch_multi on it yields the sibling paths only. */
int msgpu_tree_from_digests(msgpu_ctx* ctx, uint64_t n_classes, const uint64_t* lde_heights, const uint8_t* const* digests_dev,
                            msgpu_pdata** out, uint8_t* root32);
uint64_t msgpu_pdata_max_height(const msgpu_pdata* pd);
/* DEVICE pointer to all digest layers of a tree, back to back from the leaves up (2 * max_height - 1 digests) */
int msgpu_pdata_digests(const msgpu_pdata* pd, uint8_t** dev_ptr, uint64_t* n_digests);
/* Mmcs::commit on HOST matrices as they are (no LDE): used for the FRI layers' ExtensionMmcs rows
 * and by the parity tests of the tree shape (cases of src/types.rs:246-282). */
int msgpu_mmcs_commit(msgpu_ctx* ctx, const uint64_t* const* mats, const uint64_t* heights, const uint64_t* widths,
                      uint64_t n_mats, msgpu_pdata** out, uint8_t* root32);

void msgpu_pdata_free(msgpu_pdata* pd);
uint64_t msgpu_pdata_num_matrices(const msgpu_pdata* pd);
/* Pcs::get_evaluations_on_domain (src/prover.rs:454-468) is a view: the first rows*q stored rows of
 * matrix `idx`. Returns the device pointer and the stored shape. */
int msgpu_pdata_matrix(const msgpu_pdata* pd, uint64_t idx, uint64_t** dev_ptr, uint64_t* rows, uint64_t* cols);
/* copy stored rows [row0, row0 + nrows) of matrix idx to the host */
int msgpu_pdata_read_rows(msgpu_ctx* ctx, const msgpu_pdata* pd, uint64_t idx, uint64_t row0, uint64_t nrows,
                          uint64_t* out);
uint64_t msgpu_pdata_num_layers(const msgpu_pdata* pd);
uint64_t msgpu_pdata_layer_len(const msgpu_pdata* pd, uint64_t layer);
int msgpu_pdata_read_layer(msgpu_ctx* ctx, const msgpu_pdata* pd, uint64_t layer, uint8_t* out);
/* Mmcs::open_batch for n_idx indices at once. For query k: the opened rows of every matrix in
 * commit order (matrix m contributes stored row index >> (log_max_height - log_height_m)), written
 * back to back at opened_out + k * sum(widths); then log2(max_height) sibling digests, bottom-up,
 * at proof_out + k * 32 * log2(max_height). */
int msgpu_open_batch(msgpu_ctx* ctx, const msgpu_pdata* pd, const uint64_t* indices, uint64_t n_idx,
                     uint64_t* opened_out, uint8_t* proof_out);

/* The query phase of Pcs::open in one launch: tree k (an input commitment or a FRI commit-phase layer) is opened at
 * indices[q] >> shifts[k] for every query q. Per tree, outputs have the layout of msgpu_open_batch and follow each other:
 * opened_out gets n_idx * total_width_k values per tree, proof_out n_idx * depth_k * 32 bytes per tree. */
int msgpu_open_batch_multi(msgpu_ctx* ctx, const msgpu_pdata* const* pds, const uint32_t* shifts, uint64_t n_trees,
                           const uint64_t* indices, uint64_t n_idx, uint64_t* opened_out, uint8_t* proof_out);

/* ---- compiled constraint programs (reference `ConstraintGraph`, src/graph.rs:35-76) --------------------
 * The host compiles a circuit (src/graph.rs:120-188) and hands the flat node vector over; the library
 * lowers it to bytecode with liveness-based slot allocation for the device interpreter. */
typedef struct msgpu_program msgpu_program;
typedef struct msgpu_graph_desc {
    uint32_t n_nodes;
    const uint8_t* op;   /* 0 Const 1 Var 2 Public 3 IsFirstRow 4 IsLastRow 5 IsTransition 6 Add 7 Sub 8 Mul 9 Neg
                            (src/graph.rs:35-46) */
    const uint32_t* a;   /* Add/Sub/Mul/Neg: first child; Public: index; Var: source (0 preprocessed, 1 main,
                            2 stage 2) | row offset << 2 (0 current, 1 next)  (src/expr.rs:15-35) */
    const uint32_t* b;   /* Add/Sub/Mul: second child; Var: column index */
    const uint64_t* imm; /* Const: canonical value */
    uint32_t n_zeros;
    const uint32_t* zeros;          /* constraint roots in fold order (sorted node ids, src/graph.rs:155-156) */
    uint32_t n_lookups;
    const uint32_t* lookup_mult;    /* node id of each lookup's multiplicity */
    const uint32_t* lookup_arg_off; /* n_lookups + 1 offsets into lookup_args */
    const uint32_t* lookup_args;    /* node ids of the arguments */
    uint32_t lookup_prefix_len;     /* nodes[..lookup_prefix_len] cover the lookup expressions */
    uint32_t pre_width, main_width, stage2_width;
} msgpu_graph_desc;
/* Refuses (MSGPU_ERR_INVALID) a lookup prefix that reads a stage-2 column or a public value: lookup values are computed in
 * stage 1, before either exists. */
int msgpu_program_create(msgpu_ctx* ctx, const msgpu_graph_desc* desc, msgpu_program** out);
void msgpu_program_free(msgpu_program* prog);

/* Stage-2 (logUp accumulator) trace of one circuit, built on the device from the natural-order traces:
 * `compute_lookup_values` (src/system.rs:275-328: sweep of the lookup prefix per row, wrap-around next row)
 * + `LookupValues::stage_2_traces` (src/lookup.rs:472-555: messages beta + fingerprint(gamma, args), batch
 * inverse, exclusive running sum of multiplicity / message in (row, lookup) order, starting at zero).
 * main_dev: rows x main_width; pre_dev: rows x pre_width or NULL. stage2_out_dev: rows x stage2_width
 * (device, written). local_sum receives the circuit's total (2 u64), to be added to the running accumulator.
 * MSGPU_ERR_INVALID if a message is zero (it has no inverse). */
int msgpu_stage2_trace(msgpu_ctx* ctx, const msgpu_program* prog, const uint64_t* pre_dev, const uint64_t* main_dev,
                       uint64_t rows, const uint64_t* beta2, const uint64_t* gamma2, uint64_t* stage2_out_dev,
                       uint64_t* local_sum2);
/* Sum over claims of 1 / (beta + fingerprint(gamma, claim)) (src/prover.rs:381-387). `claims` is a HOST array of
 * n_claims x claim_len values (all claims of one length per call). out2 += is NOT applied: out2 receives the sum.
 * MSGPU_ERR_INVALID if some beta + fingerprint is zero. */
int msgpu_claims_accumulator(msgpu_ctx* ctx, const uint64_t* claims, uint64_t n_claims, uint64_t claim_len,
                             const uint64_t* beta2, const uint64_t* gamma2, uint64_t* out2);

/* The quotient stage of one circuit (src/prover.rs:437-519): evaluates the folded constraints on the
 * quotient domain GENERATOR * H_{n*q} from the committed LDEs (`quotient_values`, src/prover.rs:756-962,
 * incl. the sweep src/eval.rs:67-106, `logup_constraint_values` src/lookup.rs:152-208, selectors, the
 * reversed-alpha-power fold and the division by Z_H), then `shifted_quotient_slices` (src/prover.rs:631-679)
 * and `lde_from_shifted_coefficients` (src/prover.rs:709-717). pd_pre may be NULL. publics8 = (beta, gamma,
 * acc, next_acc) as base coordinates. Returns a device matrix of (n << log_blowup) rows x 2q columns from
 * msgpu_malloc (pass it to msgpu_commit_ldes_dev with take_ownership = 1).
 * quotient_values_out (optional, HOST, n*q*2 values) receives the quotient evaluations in natural order. */
/* Device-resident claims for one proof. Uploads n_claims x claim_len HOST values (verified canonical on the device) and
 * returns in digest32 the BLAKE3 of
 *     transcript_prefix || for each claim: le64(claim_len) || le64(value_0) || ... || le64(value_{claim_len-1})
 * i.e. of the challenger's observation buffer after the claims loop of src/prover.rs:369-372, so the host transcript
 * (`HashChallenger` flush) does not have to materialise 40 bytes per claim. The handle then serves the initial
 * accumulator (src/prover.rs:381-387) without a second copy. */
typedef struct msgpu_claims msgpu_claims;
int msgpu_claims_upload(msgpu_ctx* ctx, const uint64_t* claims, uint64_t n_claims, uint64_t claim_len,
                        const uint8_t* transcript_prefix, uint64_t prefix_len, msgpu_claims** out, uint8_t* digest32);
/* The same in two steps, so that the transfer overlaps kernels: claims_prefetch starts the host-to-device copy on the
 * context's copy stream, ordered behind everything already enqueued on the main stream (call it right after the trace
 * upload: PCIe is idle while the stage-1 LDE and Merkle kernels run); claims_digest then waits for the copy and returns the
 * digest of msgpu_claims_upload. `claims` must stay valid (pinned host memory for a real overlap) until claims_digest returns. */
int msgpu_claims_prefetch(msgpu_ctx* ctx, const uint64_t* claims, uint64_t n_claims, uint64_t claim_len, msgpu_claims** out);
int msgpu_claims_digest(msgpu_claims* cl, const uint8_t* transcript_prefix, uint64_t prefix_len, uint8_t* digest32);
int msgpu_claims_accumulate(msgpu_claims* cl, const uint64_t* beta2, const uint64_t* gamma2, uint64_t* out2);
void msgpu_claims_free(msgpu_claims* cl);

int msgpu_quotient(msgpu_ctx* ctx, const msgpu_program* prog, const msgpu_pdata* pd_pre, uint64_t idx_pre,
                   const msgpu_pdata* pd_s1, uint64_t idx_s1, const msgpu_pdata* pd_s2, uint64_t idx_s2, uint32_t log_n,
                   uint32_t log_quotient_degree, uint32_t log_blowup, const uint64_t* publics8, const uint64_t* alpha2,
                   uint64_t** lde_out_dev, uint64_t* quotient_values_out);
/* `shifted_quotient_slices` alone (host in/out; the reference's pinning test src/prover.rs:1006-1041):
 * in = nq x d quotient evaluations in natural order, out = (nq / q) x (q * d). */
int msgpu_shifted_quotient_slices(msgpu_ctx* ctx, const uint64_t* in, uint64_t nq, uint64_t d, uint64_t q, uint64_t* out);

/* ---- Pcs::open (reference src/prover.rs:580; p3-fri TwoAdicFriPcs::open + prove_fri) ------------------
 * The Fiat-Shamir transcript stays with the caller (it is generic Rust in the reference); the device does
 * the arithmetic between transcript steps:
 *   open_begin      barycentric evaluation of every column of every matrix at its points (from the first
 *                   height >> log_blowup stored rows = the coset GENERATOR * H); caller observes the values
 *   open_reduce     after alpha: per LDE height, sum over (matrix, point) of
 *                   alpha^offset * (Mred(z) - Mred(x)) / (z - x), Mred = sum_c alpha^c column_c; x in bit-reversed order
 *   fri_commit_round / fri_fold   commit phase: Merkle-commit the current vector as rows of 2 extension elements
 *                   (ExtensionMmcs: 4 base columns), then after beta fold
 *                   (1/2 + beta/2 g^-rev(i)) lo + (1/2 - beta/2 g^-rev(i)) hi and roll in the next-height input
 *                   times beta^2
 *   fri_read_current  the folded vector (for the final polynomial)
 *   fri_layer_pdata   prover data of commit-phase layer i, to answer queries with msgpu_open_batch */
typedef struct msgpu_open msgpu_open;
/* n_points[m] / points: for every matrix of every round, in order, the number of opening points and then the
 * points themselves (2 u64 each), concatenated. n_values receives the total number of extension values. */
int msgpu_open_begin(msgpu_ctx* ctx, uint64_t n_rounds, const msgpu_pdata* const* pds, const uint64_t* n_points,
                     const uint64_t* points, uint32_t log_blowup, msgpu_open** out, uint64_t* n_values);
/* opened values, order round / matrix / point / column, 2 u64 each (host buffer of 2 * n_values) */
int msgpu_open_values(msgpu_open* op, uint64_t* out);
/* builds the FRI inputs; n_inputs receives their count, log_max_height the log2 length of the first */
int msgpu_open_reduce(msgpu_open* op, const uint64_t* alpha2, uint64_t* n_inputs, uint32_t* log_max_height);
/* HOST copy of FRI input k (tallest first): 2 * len u64; len_out receives its length. Test hook. */
int msgpu_open_read_input(msgpu_open* op, uint64_t k, uint64_t* out, uint64_t* len_out);
/* sharded opening: DEVICE pointer of FRI input k (to send it to the rank that runs the commit phase), and on that rank a new
 * input of `len` extension elements to receive a peer's reduced openings into (before the first fri_commit_round; one
 * input per height) */
int msgpu_open_input_dev(msgpu_open* op, uint64_t k, uint64_t** dev_ptr, uint64_t* len_out);
int msgpu_open_add_input(msgpu_open* op, uint64_t len, uint64_t** dev_ptr);
int msgpu_fri_current_len(msgpu_open* op, uint64_t* len);
int msgpu_fri_commit_round(msgpu_open* op, uint8_t* root32);
int msgpu_fri_fold(msgpu_open* op, const uint64_t* beta2);
/* The whole commit phase with the TRANSCRIPT ON THE DEVICE, for commit_proof_of_work_bits = 0 (p3-fri `commit_phase`, reference
 * call site src/prover.rs:580): per round commit -> observe(root) -> sample beta -> fold, until the vector is stop_len long,
 * without a host round trip. input_buffer = the challenger's pending input bytes at entry (`HashChallenger` state, 1..960
 * bytes: after the alpha sample it is the 32-byte digest of the last flush). roots_out (32 bytes per round) and betas_out
 * (2 u64 per round) let the caller replay the same steps on its own challenger (and check them); max_rounds = their capacity. */
int msgpu_fri_commit_phase(msgpu_open* op, const uint8_t* input_buffer, uint64_t input_len, uint64_t stop_len, uint64_t max_rounds,
                           uint8_t* roots_out, uint64_t* betas_out, uint64_t* n_rounds);
int msgpu_fri_read_current(msgpu_open* op, uint64_t* out);
uint64_t msgpu_fri_num_layers(const msgpu_open* op);
const msgpu_pdata* msgpu_fri_layer_pdata(const msgpu_open* op, uint64_t layer);
void msgpu_open_free(msgpu_open* op);

/* ---- ONE proof over ROW SHARDS of every matrix (SURVEY 8e carried past the commitment) ---------------------------------------
 * Rank d of N holds stored rows [d H / N, (d + 1) H / N) of every committed LDE (all columns); see
 * multi_stark_b200/host/rowshard_backend.hpp for the protocol around these calls.
 * msgpu_pack_column_blocks_dev: rows x width row-major (device) -> n_blocks contiguous matrices rows x (c1[b] - c0[b]) laid out
 *   back to back in dst (the send buffer of the all-to-all that turns natural-order ROW blocks into COLUMN blocks).
 * msgpu_interleave_column_blocks_dev: the inverse for the receive side: n_blocks matrices of `rows` rows back to back in src ->
 *   one row-major rows x sum(widths) matrix.
 * msgpu_quotient_values_shard / msgpu_quotient_finish: `quotient_values` on the rows a rank holds (the NEXT rows come from the
 *   shard one trace step further) and the tail of the quotient stage on the rank that gathered the values.
 * msgpu_open_begin_shard .. msgpu_open_finish_values: Pcs::open where every rank evaluates / reduces the rows it holds; the
 *   barycentric sums are added over the ranks by the caller, the reduced-opening shards are added into the FRI owner's vectors
 *   (msgpu_open_input_dev + msgpu_ext_add_dev). Every prover data holds row shard `shard` of `n_shards` of its matrices. */
int msgpu_pack_column_blocks_dev(msgpu_ctx* ctx, const uint64_t* src, uint64_t rows, uint64_t width, uint64_t n_blocks,
                                 const uint64_t* c0, const uint64_t* c1, uint64_t* dst);
int msgpu_interleave_column_blocks_dev(msgpu_ctx* ctx, const uint64_t* src, uint64_t rows, uint64_t n_blocks, const uint64_t* widths,
                                       uint64_t* dst);
/* next_widths3 / next_col0_3 (optional): the next buffers may hold only columns [col0, col0 + width) of their matrices -- the
 * ones the constraints read at the next row (msgpu_extract_columns_dev packs them for the exchange). */
int msgpu_quotient_values_shard(msgpu_ctx* ctx, const msgpu_program* prog, const uint64_t* const* cur3, const uint64_t* const* next3,
                                const uint32_t* next_widths3, const uint32_t* next_col0_3, uint64_t row0, uint64_t n_local,
                                uint64_t next_row0, uint32_t log_n, uint32_t log_quotient_degree, const uint64_t* publics8,
                                const uint64_t* alpha2, uint64_t* out_dev);
int msgpu_extract_columns_dev(msgpu_ctx* ctx, const uint64_t* src, uint64_t rows, uint64_t width, uint64_t c0, uint64_t c1, uint64_t* dst);
int msgpu_quotient_finish(msgpu_ctx* ctx, const uint64_t* values_stored_dev, uint32_t log_n, uint32_t log_quotient_degree,
                          uint32_t log_blowup, uint64_t** lde_out_dev);
int msgpu_open_begin_shard(msgpu_ctx* ctx, uint64_t n_rounds, const msgpu_pdata* const* pds, uint32_t shard, uint32_t n_shards,
                           int fri_owner, const uint64_t* n_points, const uint64_t* points, uint32_t log_blowup,
                           msgpu_open** out, uint64_t* n_values, uint64_t* n_sums);
int msgpu_open_sums(msgpu_open* op, uint64_t* out);
int msgpu_open_finish_values(msgpu_open* op, const uint64_t* total_sums);
int msgpu_ext_add_dev(msgpu_ctx* ctx, uint64_t* dst, const uint64_t* src, uint64_t n_ext);
int msgpu_ext_add_scalar_dev(msgpu_ctx* ctx, uint64_t* v, uint64_t n_ext, const uint64_t* c2);

/* ---- peer memory over NVLink (multi_stark_b200/csrc/peer.cu) -------------------------------------------------------------------
 * The row-sharded prover's data plane without pack -> NCCL -> unpack: symmetric device windows, mapped into every rank of the node
 * with CUDA IPC, that the exchange kernels write into / read from directly (row blocks -> column blocks before the column-local
 * NTT, column blocks of the LDE -> row shards after it, subtree roots -> every peer). No counterpart in the reference
 * (single-process CPU prover); the calls replace the exchange steps of host/rowshard_backend.hpp. One process per GPU, every rank
 * makes the same calls in the same order with the same sizes (so blocks have equal (segment, offset) everywhere).
 * Growth: msgpu_peers_alloc returns 1 when no window has room; every rank then calls msgpu_peers_segment_create with the same
 * size, all-gathers the 64-byte handles over its host collective, and calls msgpu_peers_segment_open. */
#define MSGPU_MAX_PEERS 16
typedef struct msgpu_peers msgpu_peers;
int msgpu_peers_create(msgpu_ctx* ctx, int32_t rank, int32_t world, msgpu_peers** out);
int msgpu_peers_segment_create(msgpu_peers* p, uint64_t bytes, uint8_t* handle64);
int msgpu_peers_segment_open(msgpu_peers* p, const uint8_t* handles);
/* ranks inside ONE process (no IPC): bases[e] = rank e's window address (msgpu_peers_ptr of ITS object, offset 0) */
int msgpu_peers_segment_open_local(msgpu_peers* p, void* const* bases);
int msgpu_peers_alloc(msgpu_peers* p, uint64_t bytes, uint32_t* segment, uint64_t* offset);
int msgpu_peers_free_block(msgpu_peers* p, uint32_t segment, uint64_t offset);
void* msgpu_peers_ptr(const msgpu_peers* p, uint32_t segment, uint64_t offset, int32_t peer);
/* stream-ordered: work enqueued afterwards sees everything every peer wrote (and enqueued) before ITS call */
int msgpu_peers_barrier(msgpu_peers* p);
/* the 32-byte subtree root of a row-sharded commitment -> slot `rank` on every peer; *gathered_dev = world x 32 bytes (local),
 * complete after the next msgpu_peers_barrier */
int msgpu_peers_put_root(msgpu_peers* p, const uint8_t* root_dev, uint8_t** gathered_dev);
/* after a stream synchronisation: MSGPU_ERR_CUDA if a barrier timed out */
int msgpu_peers_check(msgpu_peers* p);
/* The first exchange of a row-sharded Pcs::commit (src/prover.rs:350,419 on N GPUs): row blocks -> the owners' column blocks
 * (remote stores) before the column-local LDE. The second, column blocks of the LDE -> this rank's row shard (remote loads), is
 * the leaf-hash pass of msgpu_commit_ldes_blocks_dev over msgpu_peers_ptr addresses. */
int msgpu_peers_pack_push(msgpu_peers* p, const uint64_t* src_dev, uint64_t rows, uint64_t width, uint32_t segment, uint64_t offset);
void msgpu_peers_destroy(msgpu_peers* p);

/* ---- transcript helper ---------------------------------------------------------------------------
 * Unkeyed BLAKE3-256 of a HOST byte string, hashed on the device (chunk chaining values in parallel, then the
 * binary parent tree). The reference's challenger is `HashChallenger<u8, Blake3, 32>` (src/types.rs:28-29); its
 * flush hashes the whole observation buffer, which holds 40 bytes per claim (src/prover.rs:368-373): 42 MB at
 * 2^20 claims. The digest is by definition the same as the CPU's. */
int msgpu_blake3_hash(msgpu_ctx* ctx, const uint8_t* data, uint64_t len, uint8_t* out32);

/* ---- measurement support ------------------------------------------------------------------------
 * Integer-pipe peaks of this GPU in G thread-instructions / s, from dependency-free streams timed with CUDA events:
 * out3[0] ALU pipe only (LOP3 + SHF), out3[1] FMA pipe only (IMAD), out3[2] both pipes 1 : 1. The NTT and BLAKE3
 * kernels are bound by these pipes; bench.py reports them next to the HBM roofline. */
int msgpu_measure_int_peak(msgpu_ctx* ctx, double* out3);

/* ---- test hooks --------------------------------------------------------------------------------- */
/* Bytes of the context's device memory arena in use (live msgpu_malloc blocks and everything the context's handles hold). A
 * call that leaves nothing behind, refused or complete with every handle freed, leaves this unchanged. */
int msgpu_arena_in_use(msgpu_ctx* ctx, uint64_t* bytes);
/* The selector tables of the quotient kernel: `trace_domain.selectors_on_coset(quotient_domain)` (src/prover.rs:775; p3's
 * UNNORMALISED Lagrange selectors, pinned in the reference by src/lookup.rs:697-756) at the points
 * x_i = GENERATOR * w_{n q}^i, i < n * q, in natural order. HOST outputs of n * q values each. */
int msgpu_selectors_on_coset(msgpu_ctx* ctx, uint32_t log_n, uint32_t log_q, uint64_t* is_first_row, uint64_t* is_last_row,
                             uint64_t* inv_vanishing);
/* raw 7-round BLAKE3 compression of a 16-word state and 16 message words (known-answer vector of
 * reference src/test_circuits/blake3.rs:2646-2746); host pointers */
int msgpu_blake3_compress_raw(msgpu_ctx* ctx, const uint32_t* state16, const uint32_t* msg16, uint32_t* out16);

#ifdef __cplusplus
}
#endif
#endif /* MSGPU_H */
