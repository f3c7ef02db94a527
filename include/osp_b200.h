/* osp_b200.h -- C ABI of the B200-native outer-product SpGEMM engine.
 *
 * Drop-in boundary for the functional multiply/merge path of anneouyang/OuterSPACE.
 * The reference has no FFI layer: its boundary is the C++ surface
 *
 *     size_t simulateOuterSPACE(const CSRMatrix &lmatCSC, const CSRMatrix &rmatCSR)
 *         (decl simulator/SimSpGEMM.cpp:816, def simulator/SimOuterSPACE.cpp:859)
 *
 * whose first act is `TaskProvider provider(lmatCSC, rmatCSR)` (SimOuterSPACE.cpp:860),
 * i.e. multiplyPhase (:74-97) + mergePhase (:98-132).  Every entry point below cites the
 * reference interface it replaces.  All pointers are plain pointers to the reference's
 * own storage layouts:
 *
 *     pos   = CSRMatrix::pos.data()   -- uint64_t[n_slices+1]        (common.h:41)
 *     data  = CSRMatrix::data.data()  -- packed 8-byte {uint32 idx; float val}[nnz]
 *                                                                  (common.h:10-16,42)
 *
 * No C++ or torch types cross this boundary.  Functions return OSP_OK or an error code
 * and never abort or throw (the reference asserts / throws the int 233 instead).
 * The C++ shim that keeps the reference's own names (CSRMatrix, readcoo, coo2csr<>,
 * TaskProvider) on top of this ABI is include/osp_b200.hpp.
 */
#ifndef OSP_B200_H
#define OSP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes ------------------------------------------------------------------ */
#define OSP_OK               0
#define OSP_ERR_INVALID      1   /* bad argument / k-dimension mismatch (assert, SimOuterSPACE.cpp:47) */
#define OSP_ERR_CUDA         2   /* CUDA runtime failure; osp_last_error() has the string */
#define OSP_ERR_OOM          3   /* device or host allocation failed */
#define OSP_ERR_INDEX        4   /* index out of range (assert rowId < NRow, SimOuterSPACE.cpp:68) */
#define OSP_ERR_IO           5   /* file could not be opened */
#define OSP_ERR_UNSUPPORTED  6   /* size beyond what this build handles (documented in DESIGN.md) */
#define OSP_ERR_NO_DEVICE    7   /* no CUDA device: there is NO CPU fallback */
#define OSP_ERR_DUPLICATE  233   /* duplicate (row,col); the reference throws 233 (SimSpGEMM.cpp:49) */

/* ---- flags for osp_spgemm_args.flags ------------------------------------------------- */
#define OSP_A_IS_CSR         1u  /* a_pos/a_data hold CSR(A) (a_slices = rows of A, idx = k): the engine
                                    runs the device CSR->CSC conversion (coo2csr<true>, SimSpGEMM.cpp:878) */
#define OSP_DEVICE_POINTERS  2u  /* all operand pointers are device pointers (HBM-resident operands) */
#define OSP_ROWWISE_ORDER    4u  /* the multiply emits partial products in row order of A (rows of B gathered, bins
                                    written as one stream, no task list): the default, measured faster on every config */
#define OSP_KSLICE_ORDER    32u  /* the outer-product order of the reference: k-slice after k-slice, column k of A (CSC,
                                    built on the device) against row k of B (B streamed once, bins scattered).  Same
                                    bins, same result bit for bit (DESIGN.md "multiply order") */
#define OSP_NO_FUSED_DENSE  64u  /* keep the bins even when every row is long over a small column range (see
                                    DESIGN.md "fused dense rows"): multiply -> bins -> k_merge_dense.  Without it such a
                                    product runs the bank-aligned fused kernel (k_fused_lanes, DESIGN.md K8b; environment:
                                    OSP_FUSED_LANES=0 keeps the round-1 band kernel, OSP_FL_DIRECT=0 chains the rows of C
                                    by the look-back).  Same bits. */
#define OSP_LONGROW_SWEEP  128u  /* opt-in (round 2: bit-exact on a B200, not faster than the default on config 3,
                                    profiles/r02_optin_paths.md): rows of more than 4096 partial products over more than 16384
                                    columns skip the bins -- a fused band sweep (k_long_fill, DESIGN.md section 10 item 1)
                                    computes and merges them in shared memory.  Same bits.  Ignored with
                                    OSP_KSLICE_ORDER.  Environment: OSP_LONGROW_SWEEP=1 turns it on for every call of a
                                    context, OSP_LONGROW_SWEEP_MIN=<partial products> raises the row threshold */
#define OSP_FUSED_SHORT    256u  /* opt-in (round 2: bit-exact on a B200, slower than the default, profiles/r02_chain2.md): the
                                    tiles of short rows never go through the bins -- the warp-specialised k_chain2
                                    (osp_chain2.cuh) gathers the rows of B straight into its shared-memory stages with
                                    asynchronous copies while other warps sort; k_multiply only serves the long rows.
                                    Same bits.  Ignored with OSP_KSLICE_ORDER.  Environment: OSP_FUSED_SHORT=1 */
#define OSP_NO_VALIDATE    512u  /* the caller vouches for the operand preconditions (slices ascending and duplicate-free,
                                    every column id of B below cols_b): skips the validation pass (one streaming read of
                                    both operands, k_validate).  By default a violation returns OSP_ERR_INVALID (unsorted
                                    slice, broken pos array), OSP_ERR_DUPLICATE (233) or OSP_ERR_INDEX before any merge
                                    kernel runs -- where the reference relies on coo2csr's sort + dupcheck
                                    (SimSpGEMM.cpp:113-123) */
#define OSP_KWAY_MERGE    1024u  /* rows of 4 097 .. 32 768 partial products made of at most 64 ways (runs A(i,k) * B(k,:), each
                                    sorted by construction) are merged by rank -- a k-way merge of the pre-sorted ways,
                                    the idea of merge2way / mergeHardware (SimSpGEMM.cpp:306-327, 411-441) -- instead of
                                    going through the dense accumulator of k_merge_xl.  Same bits.  Environment: OSP_KWAY=1 */
#define OSP_PROFILE_PHASES   8u  /* synchronise between phases so that stats.ms_* are per-phase times */

#define OSP_PROFILE_KERNELS 16u  /* record a CUDA-event pair around every kernel launch (osp_result_kernels) */

typedef struct osp_ctx osp_ctx;        /* one per GPU; single owner, one call at a time */
typedef struct osp_result osp_result;  /* C = A*B in HBM until freed */

/* Operands of one C = A*B.  Replaces the two `const CSRMatrix &` of simulateOuterSPACE. */
typedef struct osp_spgemm_args {
    uint64_t        a_slices;  /* a_pos has a_slices+1 entries: n_k for CSC(A), rows(A) with OSP_A_IS_CSR */
    const uint64_t *a_pos;
    const void     *a_data;    /* CSC(A): idx = row id, ascending inside a column, no duplicates */
    uint64_t        n_k;       /* inner dimension: b_pos has n_k+1 entries */
    const uint64_t *b_pos;
    const void     *b_data;    /* CSR(B): idx = col id, ascending inside a row, no duplicates */
    uint64_t        rows_c;    /* 0 = reference semantics: max row id of A + 1 (SimOuterSPACE.cpp:49-53) */
    uint64_t        cols_b;    /* 0 = derive as max col id of B + 1; otherwise every col id must be < cols_b */
    uint32_t        flags;
    uint32_t        reserved;
    uint64_t        a_nnz;     /* OSP_DEVICE_POINTERS only: a_pos[a_slices] and b_pos[n_k] when the caller knows them */
    uint64_t        b_nnz;     /* (saves a device->host read at the start of the call); 0 = read them from the device */
} osp_spgemm_args;

/* Counters of one call (all sizes in elements, times in milliseconds of device time). */
typedef struct osp_stats {
    uint64_t rows_c, cols_b, n_k;
    uint64_t nnz_a, nnz_b, nnz_c;
    uint64_t products;            /* P = sum_k nnz(A(:,k))*nnz(B(k,:)) = mulflops_ref, SimSpGEMM.cpp:884-891 */
    uint64_t algorithmic_bytes;   /* SURVEY.md 8d: 16P + 8nnzC + 24nnzA + 8nnzB + 8(2m+3n+5) */
    uint64_t merge_tiles;         /* tiles of consecutive rows the merge kernel took */
    uint64_t rows_medium;         /* rows sorted by one CTA in shared memory (512 < partial products <= 4096) */
    uint64_t rows_long;           /* rows folded through a dense accumulator (> 4096 partial products) */
    uint64_t kernel_launches;     /* kernels this call launched */
    uint64_t row_chunks;          /* output-row blocks the call was split into */
    float    ms_total;            /* first kernel to last kernel */
    float    ms_convert;          /* CSR->CSC conversion + symbolic count/scan */
    float    ms_multiply;
    float    ms_merge;
    float    ms_h2d, ms_d2h;      /* host-pointer calls only */
    float    ms_exchange;         /* osp_dist_spgemm: the all-to-allv of partial products */
    float    reserved_f;
    uint64_t exchange_bytes_out;  /* osp_dist_spgemm: bytes of partial products this rank sent to other ranks */
} osp_stats;

/* ---- context ------------------------------------------------------------------------- */
int  osp_device_count(void);                        /* 0 when no usable GPU */
int  osp_create(int device, osp_ctx **out);         /* binds to one GPU, creates its stream + workspace */
void osp_destroy(osp_ctx *ctx);
const char *osp_last_error(const osp_ctx *ctx);     /* message of the last failing call on ctx (or global) */
int  osp_set_workspace_limit(osp_ctx *ctx, uint64_t bytes); /* cap on partial-product workspace; larger
                                                       products are processed in output-row blocks */
int  osp_set_result_limit(osp_ctx *ctx, uint64_t bytes);    /* cap on the up-front allocation of C's data; 0 (default) =
                                                       what the device can spare.  C is allocated at the plan's bound
                                                       sum_i min(partials of row i, cols) when that fits; otherwise at the
                                                       cap, and the call runs in row blocks, each admitted against the cap
                                                       with the exact nnz(C) so far (OSP_ERR_OOM when a block cannot fit) */
void *osp_stream(osp_ctx *ctx);                     /* the cudaStream_t every kernel of ctx runs on */

/* ---- the hot path: TaskProvider(lmatCSC, rmatCSR) ------------------------------------- */
int  osp_spgemm(osp_ctx *ctx, const osp_spgemm_args *args, osp_result **out);
int  osp_result_dims(const osp_result *r, uint64_t *rows, uint64_t *nnz);
int  osp_result_copy(osp_result *r, uint64_t *pos, void *data);  /* into CSRMatrix::pos / ::data storage */
/* Rows [row_begin, row_end) of C: pos gets row_end - row_begin + 1 absolute offsets into C's data, data the
 * pos[last] - pos[0] elements of those rows (data = NULL: offsets only, to size the buffer).  For results larger than
 * the caller's host memory (config 3 at full scale holds tens of GB of C). */
int  osp_result_copy_rows(osp_result *r, uint64_t row_begin, uint64_t row_end, uint64_t *pos, void *data, uint64_t data_capacity);
int  osp_result_device(const osp_result *r, const uint64_t **d_pos, const void **d_data);
int  osp_result_stats(const osp_result *r, osp_stats *stats);
/* Per-launch device times of a call made with OSP_PROFILE_KERNELS, in launch order (two-call pattern:
 * pass names = ms = NULL to get the count in *n; then arrays of *n entries).  Names are static strings. */
int  osp_result_kernels(const osp_result *r, uint64_t *n, const char **names, float *ms);
void osp_result_free(osp_result *r);

/* Task-size lists the reference's timing models read from TaskProvider
 * (getMultiplyTasks/getMergeTasks, SimOuterSPACE.cpp:59-64; MultiplyTask/MergeTask :34-42):
 * per non-empty k-slice (nnzc, nnzr), and per output row (#ways, output nnz).
 * (nnzc, nnzr) and #ways equal the as-written TaskProvider's; "output nnz" is the true number of non-zeros of the row
 * of C (intended semantics) -- the as-written merge counts 1 + the adjacent equal position-index pairs there because of
 * its inverted duplicate test (SimOuterSPACE.cpp:120), which this engine does not reproduce.
 * Two-call pattern: pass NULL arrays to obtain the counts. */
int  osp_task_sizes(osp_ctx *ctx, const osp_spgemm_args *args, const osp_result *r,
                    uint64_t *n_multiply, uint32_t *multiply_nnzc_nnzr,
                    uint64_t *n_merge, uint32_t *merge_ways_out);

/* ---- k-sharded multi-GPU path: one process (and one osp_ctx) per GPU ------------------------ */
/* The reference is single-process; BASELINE.json north_star adds: each GPU runs the outer products of
 * its k-range (TaskProvider::multiplyPhase, SimOuterSPACE.cpp:74-97, restricted to k0 <= i < k1), partial
 * products travel to the owner of their output row with an NCCL all-to-allv, owners merge
 * (mergePhase, :98-132).  Owners are contiguous row blocks [rows*r/world, rows*(r+1)/world). */
typedef struct osp_dist osp_dist;
int  osp_dist_unique_id(void *id128);               /* ncclGetUniqueId: 128 bytes, made on one rank, given to all */
int  osp_dist_create(osp_ctx *ctx, const void *id128, int rank, int world, osp_dist **out);
void osp_dist_destroy(osp_dist *d);
int  osp_dist_rows(const osp_dist *d, uint64_t rows_c, uint64_t *row_begin, uint64_t *row_end);
/* args = this rank's shard: CSR(A[:, k0:k1]) with k ids relative to k0 (OSP_A_IS_CSR required; a_slices
 * <= rows_c rows), CSR(B[k0:k1, :]) with n_k = k1 - k0; rows_c and cols_b = dimensions of C (required,
 * the same on every rank).  Collective: every rank of the communicator must call it.  *out holds this
 * rank's rows [row_begin, row_end) of C, bit-identical to the single-GPU result. */
int  osp_dist_spgemm(osp_dist *d, const osp_spgemm_args *args, osp_result **out);

/* ---- device CSR->CSC of one operand: coo2csr<true> (SimSpGEMM.cpp:111-117,878) -------- */
/* Stable: inside an output slice the source slice ids ascend.  pos_out[n_minor+1], data_out[nnz].
 * flags: OSP_DEVICE_POINTERS or 0.  A bit-exact permutation of the input (NaN payloads included).  A duplicate
 * (slice, id) pair is OSP_ERR_DUPLICATE; an id >= n_minor is OSP_ERR_INDEX, so is any entry when n_minor = 0.
 * Limit: the slices are sorted with the merge machinery of osp_spgemm, source slice ids as the column ids.  An output
 * slice of more than 512 entries (more than 4096 once n_major exceeds 131072) borrows the long-row accumulator of
 * 4 * n_major bytes + a bitmap, which must fit in max(1/16 of the device, 256 MB); otherwise the call is
 * OSP_ERR_UNSUPPORTED ("column range too large"), e.g. n_major = 2^32 - 1 with a slice of 5000 entries on a B200. */
int  osp_csr2csc(osp_ctx *ctx, uint64_t n_major, uint64_t n_minor, const uint64_t *pos, const void *data,
                 uint32_t flags, uint64_t *pos_out, void *data_out);

/* ---- host loaders (the reference's .mtx surface) -------------------------------------- */
typedef struct osp_coo osp_coo;
int  osp_readcoo(const char *path, int symmetric, osp_coo **out);          /* readcoo, SimSpGEMM.cpp:55-100 */
int  osp_readcoo_buffer(const char *text, uint64_t len, int symmetric, osp_coo **out);  /* same, text in memory (the
                                                                reference's readcoo takes a std::istream) */
int  osp_coo_dims(const osp_coo *c, uint64_t *nrow, uint64_t *ncol, uint64_t *nnz);
int  osp_coo_copy(const osp_coo *c, uint32_t *rows, uint32_t *cols, float *vals);
void osp_coo_free(osp_coo *c);
/* coo2csr<transpose> + dupcheck (SimSpGEMM.cpp:43-53,102-152): pos[N+1], data[nnz]. */
int  osp_coo2csr(uint64_t nnz, const uint32_t *rows, const uint32_t *cols, const float *vals,
                 uint64_t N, int transpose, uint64_t *pos, void *data);

/* Compact COO (CompactCOOMatrix, common.h:52-56; the reference's alternative operand format for the multiply,
 * compactMulcsr SimSpGEMM.cpp:247-263).  Triplets are returned as three arrays like osp_coo_copy.
 * osp_csr2compact = csr2compact (SimSpGEMM.cpp:154-219): group j = the (j+1)-th non-zero of every slice that has
 * one, slices ascending; *n_groups = the longest slice.  Call with group_pos = NULL for n_groups alone, then with
 * group_pos[n_groups + 1] and rows/cols/vals[nnz].  A matrix without non-zeros has 0 groups (undefined behaviour in
 * the reference).  osp_csc2rawcompact = csc2rawcompact (SimSpGEMM.cpp:221-243): one group per slice (group_pos =
 * pos), row = the element's index, col = the slice id.
 * A compact operand enters the engine as the triplet list it is: osp_coo2csr_device(rows, cols, vals) -> osp_spgemm
 * gives the merged equivalent of compactMulcsr (tests/test_compact.py). */
int  osp_csr2compact(uint64_t n_major, const uint64_t *pos, const void *data, uint64_t *n_groups, uint64_t *group_pos,
                     uint32_t *rows, uint32_t *cols, float *vals);
int  osp_csc2rawcompact(uint64_t n_major, const uint64_t *pos, const void *data, uint32_t *rows, uint32_t *cols, float *vals);

/* The same conversion on the GPU (histogram -> scan -> bucket scatter -> per-slice sort with the merge machinery;
 * a slice that shrinks while folding held a duplicate -> OSP_ERR_DUPLICATE = the reference's throw(233)).
 * N = number of slices (rows for CSR, columns when transpose); n_other = range of the other index (0 = derive it;
 * required with device pointers).  flags: OSP_DEVICE_POINTERS (triplet arrays and outputs in HBM) or 0.
 * N = 0 with triplets is OSP_ERR_INDEX.  Same limit as osp_csr2csc with n_other in place of n_major: a slice of more
 * than 4096 triplets with n_other = 2^32 - 1 is OSP_ERR_UNSUPPORTED on a B200. */
int  osp_coo2csr_device(osp_ctx *ctx, uint64_t nnz, const uint32_t *rows, const uint32_t *cols, const float *vals,
                        uint64_t N, uint64_t n_other, int transpose, uint32_t flags, uint64_t *pos, void *data);

/* .mtx ingest on the device: the text of a file (or of the caller's memory) goes to HBM once and is parsed there into
 * the triplets osp_readcoo gives -- the same entries in the same order with the same float bits, the same errors
 * (OSP_ERR_INVALID for a line that is no entry, blank line or comment; osp_last_error names its line).  The resulting
 * osp_coo keeps its triplets in the device memory of ctx (SoA: rows, cols, vals) and must be freed before ctx.
 * osp_coo_dims, osp_coo_copy (to the host) and osp_coo_free take it like a host osp_coo.  The text and 12 bytes per
 * line must fit the device together (OSP_ERR_OOM otherwise, and ctx stays usable); 2^32 or more entries is
 * OSP_ERR_UNSUPPORTED. */
int  osp_readcoo_device(osp_ctx *ctx, const char *path, int symmetric, osp_coo **out);
int  osp_readcoo_buffer_device(osp_ctx *ctx, const char *text, uint64_t len, int symmetric, osp_coo **out);
int  osp_coo_device(const osp_coo *c, const uint32_t **rows, const uint32_t **cols, const float **vals); /* OSP_ERR_INVALID for a host coo */
/* coo2csr<transpose> + dupcheck of a device-resident osp_coo into a device CSR of N slices: the bytes and the errors of
 * osp_coo2csr (OSP_ERR_DUPLICATE, OSP_ERR_INDEX for an id >= N).  The range of the other index is the largest id the
 * ingest recorded + 1.  *out is a result like osp_bias_relu's: osp_result_device gives an operand for
 * osp_spgemm(OSP_DEVICE_POINTERS | ...), osp_result_copy the host CSRMatrix.  Same limit as osp_coo2csr_device. */
int  osp_coo2csr_result(osp_ctx *ctx, const osp_coo *c, uint64_t N, int transpose, osp_result **out);

/* ---- layer chaining: relu(C + bias) kept sparse ------------------------------------------------------------- */
/* What a layer of the reference's MLP applies between two products (x = relu(fc(x)), NN_models/models.py:18-31):
 * out(i,c) = C(i,c) + bias[c] (one rounded fp32 add; bias[c] alone where C has no entry), kept where > 0.
 * bias: cols floats (host, or device with OSP_DEVICE_POINTERS), NULL = no bias (then only C's entries > 0 stay).
 * 1 <= cols <= 16384 (the row is densified in shared memory).  *out is a new result: its device CSR
 * (osp_result_device) is the A operand of the next layer's osp_spgemm (OSP_A_IS_CSR | OSP_DEVICE_POINTERS). */
int  osp_bias_relu(osp_ctx *ctx, const osp_result *c, uint64_t cols, const float *bias, uint32_t flags, osp_result **out);

const char *osp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* OSP_B200_H */
