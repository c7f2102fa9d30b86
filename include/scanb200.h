/*
 * scanb200.h -- C ABI of the B200-native normalize -> PCA path of scan-rs.
 *
 * This is the drop-in boundary (SURVEY.md 8b): plain pointers and sizes, opaque handles,
 * int status codes, no C++/torch types.  A Rust crate binds exactly these symbols from
 * its build.rs (INTEGRATION.md shows the `extern "C"` block and the safe wrappers that
 * keep the reference's entry points: `AdaptiveMat` -> upload, `normalize(..)`,
 * `Pca::run_pca_cancellable`).  Each entry point cites the reference interface it
 * replaces (paths relative to the reference checkout).
 *
 * Conventions
 *   - Matrix orientation is the reference's: features/genes are ROWS, barcodes/cells are
 *     COLUMNS (scan-rs/src/mtx.rs:10-51).  m = genes, n = cells.
 *   - All dense blocks are row-major ("standard layout" of ndarray), f64.
 *   - Host buffers are caller-allocated and caller-owned; the library never keeps a host
 *     pointer after the call returns.  Handles own device memory.
 *   - One sb_ctx drives one GPU from one host thread.  For cell-sharded multi-GPU runs
 *     every rank (one process per GPU) creates its own context, joins a communicator
 *     with sb_comm_init and then makes the SAME sequence of calls on its own cell shard;
 *     gene-sized results (totals, U, sigma) come back replicated, cell-sized results
 *     (cell totals, V) come back for the local shard only.
 *   - Every function returns SB_OK (0) or an error code; sb_last_error() returns the
 *     thread-local message.  Nothing panics or aborts across the ABI.
 *   - There is NO CPU fallback: without a CUDA device sb_init fails with SB_ERR_CUDA.
 */
#ifndef SCANB200_H
#define SCANB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB_VERSION 100

#if defined(__GNUC__)
#define SB_API __attribute__((visibility("default")))
#else
#define SB_API
#endif

/* status codes */
enum {
    SB_OK = 0,
    SB_ERR_INVALID_SHAPE = 1, /* "The input matrix must be at least 2x2."  bk_svd.rs:73-75 */
    SB_ERR_INVALID_K = 2,     /* "invalid k"                                 bk_svd.rs:77-79 */
    SB_ERR_CANCELLED = 3,     /* snoop::CancellationError                    snoop/src/lib.rs:5-18 */
    SB_ERR_CUDA = 4,
    SB_ERR_NCCL = 5,
    SB_ERR_OOM = 6,
    SB_ERR_INVALID_ARG = 7,   /* the reference's assert!/panic! programmer errors */
    SB_ERR_UNSUPPORTED = 8,
    SB_ERR_LINALG = 9         /* cuSOLVER failure (the reference's LAPACK `?` errors) */
};

/* storage order of host CSR/CSC arrays handed to sb_upload (sprs::CSR / sprs::CSC of a
 * genes x cells matrix, sqz/src/mat.rs:45-65) */
enum { SB_GENE_MAJOR = 0, SB_CELL_MAJOR = 1 };

/* scan_rs::normalization::Normalization (scan-rs/src/normalization.rs:11-28) */
enum {
    SB_NORM_CELLRANGER = 0,
    SB_NORM_CELLRANGER8 = 1,
    SB_NORM_SEURATLOG = 2,
    SB_NORM_BINOMIAL_DEVIANCE = 3,
    SB_NORM_BINOMIAL_PEARSON = 4,
    SB_NORM_WITH_SIZE_FACTORS = 5,
    SB_NORM_LOG_TRANSFORM = 6
};

/* scan_rs::normalization::LogBase (normalization.rs:105-112) */
enum { SB_LOG_E = 1, SB_LOG_TWO = 2, SB_LOG_TEN = 10 };

typedef struct sb_ctx sb_ctx;   /* device context (+ optional NCCL communicator) */
typedef struct sb_mat sb_mat;   /* device-resident u32 count matrix: AdaptiveMat<u32> (sqz/src/mat.rs:34-42) */
typedef struct sb_nmat sb_nmat; /* normalized matrix: LowRankOffset<D, impl MatrixMap<u32,f64>> (sqz/src/low_rank_offset.rs:12-16) */

/* progress / cancel token: CancelProgress::set_progress_check (snoop/src/lib.rs:45-57).
 * Called on the calling thread with the reference's milestones (0.8*i/n_iter, 0.82, 0.93,
 * 1.0; bk_svd.rs:96-114).  A non-zero return cancels: the call stops at that milestone and
 * returns SB_ERR_CANCELLED. */
typedef int (*sb_progress_cb)(double fraction, void *user);

/* ---------------------------------------------------------------- context */
SB_API int sb_version(void);
SB_API const char *sb_last_error(void);
SB_API int sb_init(int device, sb_ctx **out);
SB_API void sb_shutdown(sb_ctx *ctx);
/* Multi-GPU: rank 0 calls sb_comm_unique_id, ships the 128 bytes to the other ranks by any
 * means (torch.distributed, MPI, a file), then every rank calls sb_comm_init. */
SB_API int sb_comm_unique_id(char id[128]);
SB_API int sb_comm_init(sb_ctx *ctx, int nranks, int rank, const char id[128]);
SB_API int sb_sync(sb_ctx *ctx);
/* One host thread, every GPU of the box (SURVEY 8b: the reference's caller is a single process, tools/src/bin/cmd.rs:67-81).
 * sb_multi_init creates one context per device (devices == NULL: 0..n-1), joins them to one communicator and starts one worker
 * thread per device.  sb_multi_run executes fn(rank, ctx, user) on every worker concurrently and returns when all are done (the
 * first non-zero status, with "rank r: message" as the error): inside fn each rank makes the ordinary single-context calls on
 * its own cell shard, exactly the sequence one-process-per-GPU callers make.  Handles created inside fn stay valid across
 * sb_multi_run calls and must be freed before sb_multi_shutdown. */
typedef struct sb_multi sb_multi;
typedef int (*sb_rank_fn)(int rank, sb_ctx *ctx, void *user);
SB_API int sb_multi_init(int n, const int *devices, sb_multi **out);
SB_API int sb_multi_size(const sb_multi *mm);
SB_API int sb_multi_ctx(sb_multi *mm, int rank, sb_ctx **out);
SB_API int sb_multi_run(sb_multi *mm, sb_rank_fn fn, void *user);
SB_API void sb_multi_shutdown(sb_multi *mm);
/* Options: "direct_projection" (0/1, default 0): 1 forces the wide projection pass T = Q^T A of
 * bk_svd.rs:102,131 to run as a sparse product; 0 lets the library use Q^T A = R^-T (K^T A) when R is usable.
 * "gather" (default 1): 1 = panelled gather kernels for the sparse halves of both products, 0 = the first-generation
 * cell-major / gene-major kernels (A/B and accuracy reference).  "dense_genes" (default 2048) / "dense_min_density"
 * (default 0.12): size of the dense hot-gene panel of matrices uploaded afterwards (0 disables it).
 * "upload_sync" (default 1): drain the build stream after every stage of a pipelined upload.
 * "overlap" / "overlap_t" (default 0): experimental concurrent sparse + panel kernels.
 * "dense_max_count" (default 15, 1..15): largest count kept in the dense panel of matrices uploaded afterwards.
 * "gather_split" (default 0): EXPERIMENTAL separate 4-byte stream for the sparse entries with a count of 1 (gather_split.cu);
 * written without hardware access, off until validated.
 * "panel_i8" (default 0): EXPERIMENTAL tcgen05 int8 contraction of the T-side panel (needs dense_max_count <= 3, a
 * 2,048-gene panel and width <= 20); written without hardware access, off until validated. */
SB_API int sb_set_option(sb_ctx *ctx, const char *name, double value);

/* Page-locked host memory for inputs / outputs (optional): copies to and from pinned buffers run at PCIe
 * speed and asynchronously; pageable buffers work too, several times slower for the large V block. */
SB_API int sb_host_alloc(size_t bytes, void **out);
SB_API void sb_host_free(void *p);

/* ---------------------------------------------------------------- count matrix
 * sb_upload replaces AdaptiveMat::from_csmat / new (sqz/src/mat.rs:81-124): the Rust side
 * decodes each AdaptiveVec once (vec.rs `foreach` :1230-1273) into these arrays.  `major`
 * says whether indptr runs over genes (idx = cell) or over cells (idx = gene).  n_local is
 * this rank's number of cells.  Indices must be strictly ascending inside each vector and
 * counts non-zero (what AdaptiveVec guarantees); zeros are dropped. */
SB_API int sb_upload(sb_ctx *ctx, int major, uint32_t m, uint64_t n_local, const uint64_t *indptr,
              const uint32_t *idx, const uint32_t *cnt, sb_mat **out);
/* The reference's own storage as upload input: one AdaptiveVec (sqz/src/vec.rs:1029-1053) described by the raw parts of its Rust
 * struct.  variant follows the enum order: 0 D3, 1 D4, 2 D8, 3 D16, 4 V, 5 S3, 6 S4, 7 S8.
 *   D3/D4/D8/D16 : dense = Dense3.data (u64 words, 21 x 3 bits) / Dense4.data (bytes, 2 x 4 bits) / DenseW.data (u8 / u16), one code
 *                  per position; fb_* = the SimpleSparse fallback holding the values the narrow code cannot (vec.rs:660-1023)
 *   V            : fb_* = SimpleSparse.indexes / values (vec.rs:123-127); dense unused
 *   S3/S4/S8     : CompressedIndexSparse (vec.rs:222-227): index_bytes[n_index] (position inside a block of 256), block_starts
 *                  [n_block_starts]; dense / fb_* describe its dense_data (a D3 / D4 / D8 vector of length n_index)
 * len = the vector's logical length.  All arrays stay owned by the caller. */
typedef struct sb_adaptive_vec {
    uint32_t variant;
    uint32_t reserved;
    uint64_t len;
    const void *dense;
    const uint32_t *fb_idx;
    const uint32_t *fb_val;
    uint64_t fb_len;
    const uint8_t *index_bytes;
    uint64_t n_index;
    const uint32_t *block_starts;
    uint64_t n_block_starts;
} sb_adaptive_vec;
/* AdaptiveVec::foreach (vec.rs:1230-1273) for one vector: (index, value) ascending, stored zeros skipped.  idx / val may be NULL
 * to count only. */
SB_API int sb_adaptive_decode_vec(const sb_adaptive_vec *vec, uint32_t *idx, uint32_t *val, uint64_t capacity, uint64_t *nnz);
/* AdaptiveMat (sqz/src/mat.rs:34-42) -> device matrix: decodes the m (SB_GENE_MAJOR, the reference's CSR storage) or n_local
 * (SB_CELL_MAJOR) vectors on `threads` host threads (0 = all) and uploads. */
SB_API int sb_upload_adaptive(sb_ctx *ctx, int major, uint32_t m, uint64_t n_local, const sb_adaptive_vec *vecs, int threads,
                       sb_mat **out);
/* The same constructor for a cell-major matrix in a narrow host form, for m <= 65536: u16 gene index + u8 count per entry
 * (3 bytes over PCIe instead of 8 -- the host-to-device copy is the largest part of an end-to-end call).  Counts >= 255
 * are written as 255 in cnt8 and listed in the side arrays: entry big_pos[i] (ascending stream positions) has count
 * big_cnt[i].  The Rust side fills these from the same AdaptiveVec `foreach` walk (vec.rs:1230-1273) as sb_upload's. */
SB_API int sb_upload_compact(sb_ctx *ctx, uint32_t m, uint64_t n_local, const uint64_t *indptr, const uint16_t *idx16,
                      const uint8_t *cnt8, uint64_t n_big, const uint64_t *big_pos, const uint32_t *big_cnt, sb_mat **out);
/* The same constructor in the packed host form -- about 1.55 bytes per entry over PCIe (the compact form: 3, the plain one: 8),
 * for any m the library accepts.  Per entry, in the stream order of sb_upload's cell-major arrays:
 *   dgene[j]  : gene - previous gene of the same cell (the previous gene of a cell's first entry is -1), if that is in 1..255;
 *               else 0, and (j, gene) is appended to esc_pos / esc_gene (stream positions ascending)
 *   cnt4[j/2] : count in the low (j even) or high (j odd) nibble, if below 15; else 15, and (j, count) is appended to big_pos /
 *               big_cnt (ascending).  cnt4 has (nnz + 1) / 2 bytes.
 * The Rust side fills these from the same AdaptiveVec `foreach` walk (vec.rs:1230-1273); sb_pack_csc_count / sb_pack_csc_fill do it
 * from plain cell-major u32 arrays on `threads` host threads (0 = all): _count returns the two side-list lengths, _fill writes
 * every array (all caller-allocated; page-locked memory from sb_host_alloc makes the upload a straight DMA).  A zero delta without
 * an escape record, or an escaped gene that does not ascend inside its cell, is SB_ERR_INVALID_ARG. */
SB_API int sb_pack_csc_count(uint64_t n, const uint64_t *indptr, const uint32_t *idx, const uint32_t *cnt, int threads, uint64_t *n_esc,
                      uint64_t *n_big);
SB_API int sb_pack_csc_fill(uint64_t n, const uint64_t *indptr, const uint32_t *idx, const uint32_t *cnt, int threads, uint8_t *dgene,
                     uint8_t *cnt4, uint64_t *esc_pos, uint32_t *esc_gene, uint64_t *big_pos, uint32_t *big_cnt);
SB_API int sb_upload_packed(sb_ctx *ctx, uint32_t m, uint64_t n_local, const uint64_t *indptr, const uint8_t *dgene, const uint8_t *cnt4,
                     uint64_t n_esc, const uint64_t *esc_pos, const uint32_t *esc_gene, uint64_t n_big, const uint64_t *big_pos,
                     const uint32_t *big_cnt, sb_mat **out);
/* The loaders' device half (SURVEY 8f rank 2).  sb_upload_unsorted: cell-major arrays whose gene indices are in ANY order inside
 * a cell -- the Cell Ranger 3 defect that hdf5-io/src/matrix.rs:63-78 repairs with `new_from_unsorted_csc`; every cell's entries
 * are sorted on the device, a duplicate index inside a cell is SB_ERR_INVALID_ARG.  sb_filter_genes: compute_genes_filter + the
 * row selection of read_adaptive_csr_matrix (matrix.rs:93-192): type_keep[m] (NULL = all) marks the features whose type matches
 * `retain_feature_like`, min_total is `shrink_row`; kept_rows (room for m) receives the survivors in file order. */
SB_API int sb_upload_unsorted(sb_ctx *ctx, uint32_t m, uint64_t n_local, const uint64_t *indptr, const uint32_t *idx,
                       const uint32_t *cnt, sb_mat **out);
SB_API int sb_filter_genes(sb_mat *mat, const uint8_t *type_keep, uint64_t min_total, uint32_t *kept_rows, uint32_t *n_kept,
                    sb_mat **out);
/* rows(), cols(), shape() (mat.rs:160-176) + nnz() (:155-157); n_global == n_local without a communicator */
SB_API int sb_mat_shape(const sb_mat *mat, uint32_t *m, uint64_t *n_local, uint64_t *n_global, uint64_t *nnz_local);
/* to_csmat (mat.rs:207-239): sizes from sb_mat_shape; indptr has m+1 or n_local+1 entries */
SB_API int sb_download(const sb_mat *mat, int major, uint64_t *indptr, uint32_t *idx, uint32_t *cnt);
SB_API void sb_free_mat(sb_mat *mat);

/* sum_axis::<u32>(Axis(0)) (mat.rs:377-406; normalization.rs:159,161): per-cell UMI totals, wrapping u32 */
SB_API int sb_cell_totals(sb_mat *mat, uint32_t *out_n_local);
/* per-gene totals as u64 (hdf5-io/src/matrix.rs:106-114; sum_axis(Axis(1))); all-reduced over ranks.
 * square != 0 gives sum of v*v (HVG moments, builder-defined, SURVEY 8c) */
SB_API int sb_gene_totals(sb_mat *mat, int square, uint64_t *out_m);
/* number of stored non-zeros per gene, all-reduced */
SB_API int sb_gene_nnz(sb_mat *mat, uint64_t *out_m);
/* median_mut over the cell totals of ALL ranks (scan-rs/src/stats.rs:13-38): u32 midpoint.
 * *nonempty = 0 when there are no cells (the caller then uses 1.0, normalization.rs:166) */
SB_API int sb_median_cell_total(sb_mat *mat, uint32_t *median, int *nonempty);

/* partition_on_thresholds (mat.rs:772-889).  `rows_out`/`cols_out` need room for m / n_local entries and receive the
 * selected indices; kept/residual may be NULL.  Sharded contexts: gene sums are all-reduced every round, cell verdicts stay
 * local; cols_out are LOCAL cell indices and the returned matrices hold this rank's shard. */
SB_API int sb_partition(sb_mat *mat, int has_row_thr, double row_thr, int has_col_thr, double col_thr,
                 sb_mat **kept, sb_mat **residual, uint64_t *rows_out, uint64_t *n_rows_out,
                 uint64_t *cols_out, uint64_t *n_cols_out);
/* select_rows / select_cols (mat.rs:1004-1071): new matrix with the given rows/cols in the given order (sharded contexts:
 * every rank passes the same rows; cols are LOCAL cell indices of its own shard) */
SB_API int sb_select_rows(sb_mat *mat, const uint32_t *rows, uint32_t count, sb_mat **out);
SB_API int sb_select_cols(sb_mat *mat, const uint64_t *cols, uint64_t count, sb_mat **out);
/* Highly-variable-gene selection (NOT in the reference; builder-defined, SURVEY 8c): exact u64
 * sums -> dispersion var/mean in f64 -> top n_top, ties to the lower index; out sorted ascending. */
SB_API int sb_hvg_select(sb_mat *mat, uint32_t n_top, uint32_t *out_idx, uint32_t *out_count);

/* ---------------------------------------------------------------- normalization
 * normalize / normalize_with_size_factor (normalization.rs:46-102) plus the two binomial
 * residual constructors the CLI dispatches to (normalization.rs:233-260, 307-323;
 * tools/src/bin/cmd.rs:67-81).  size_factors (u32[n_local]) only for SB_NORM_WITH_SIZE_FACTORS.
 * The result borrows `mat`: free it before the matrix. */
SB_API int sb_normalize(sb_mat *mat, int norm, const uint32_t *size_factors, sb_nmat **out);
/* log_normalize_with_size_factor (+ optional scale_and_center) with every knob exposed
 * (normalization.rs:138-178; mat.rs:986-1001): has_target=0 -> median of cell totals;
 * center_scale: 0 = sparse log-normalized matrix only, 1 = scale_and_center(Axis(1), None),
 * 2 = scale_and_center(Axis(1), Some(sd_override[m])). */
SB_API int sb_log_normalize(sb_mat *mat, int has_target, double target, int log_base, const uint32_t *size_factors,
                     int center_scale, const double *sd_override, sb_nmat **out);
/* log1p_normalize_fixed_point (normalization.rs:191-213) */
SB_API int sb_normalize_fixed_point(sb_mat *mat, int log_base, uint32_t base, uint32_t exponent, sb_nmat **out);
/* The derived tables: col_scale[n_local], row_scale[m] (1/sd), u[m], v[n_local]; any pointer may be NULL */
SB_API int sb_nmat_params(const sb_nmat *a, double *col_scale, double *row_scale, double *u, double *v);
/* LowRankOffset::to_dense (low_rank_offset.rs:55-57): m x n_local row-major; test/debug sizes only */
SB_API int sb_nmat_to_dense(sb_nmat *a, double *out);
/* LowRankOffset . Array2 (low_rank_offset.rs:68-81): out[m x w] = A . x[n_local x w], all-reduced over ranks */
SB_API int sb_nmat_dot(sb_nmat *a, const double *x, uint32_t w, double *out);
/* Array2 . LowRankOffset (low_rank_offset.rs:83-96): out[w x n_local] = b[w x m] . A */
SB_API int sb_nmat_rdot(sb_nmat *a, const double *b, uint32_t w, double *out);
/* Squared Frobenius norm of the normalized matrix (offset included): the denominator of the DERIVED "variance explained"
 * sigma_i^2 / ||A||_F^2.  Not part of the reference's result (PcaResult is (u, d, v), dim_red/mod.rs:47); north_star names it,
 * so it is offered as a labelled convenience.  Log-chain normalizations only (SB_ERR_UNSUPPORTED otherwise). */
SB_API int sb_nmat_frobenius_sq(sb_nmat *a, double *out);
SB_API void sb_free_nmat(sb_nmat *a);

/* ---------------------------------------------------------------- PCA
 * The start block: SmallRng::seed_from_u64(seed) + Uniform::new(-1.0, 1.0), row-major fill
 * (bk_svd.rs:83-84, :90, :118).  Host-side, deterministic. */
SB_API int sb_omega(uint64_t seed, uint64_t rows, uint64_t cols, double *out);

/* svd_bk (scan-rs/src/dim_red/bk_svd.rs:57-146).  b is clamped to min(m, n, b) (:81).  `omega`
 * may be NULL (generated from `seed` as above) or the caller's start block, row-major:
 * (b x m) when n > m, (n_local x b) when m >= n.  Outputs: U[m x k], S[k], V[n_local x k]
 * row-major -- V is already `vt.reversed_axes()` as run_pca returns it (bk_svd.rs:51). */
SB_API int sb_bksvd(sb_nmat *a, uint32_t k, uint32_t b, uint32_t n_iter, uint64_t seed, const double *omega,
             sb_progress_cb cb, void *user, double *U, double *S, double *V);
/* BkSvd::run_pca_cancellable (bk_svd.rs:48-52): b = ceil(k * k_multiplier), seed 0 */
SB_API int sb_bksvd_run_pca(sb_nmat *a, uint32_t k, double k_multiplier, uint32_t n_iter, sb_progress_cb cb,
                     void *user, double *U, double *S, double *V);
/* Diagnostics of the last sb_bksvd on this context: the condition estimate of the Krylov basis' triangular factor that gated the
 * projection identity (0 when the direct pass ran unconditionally), the a-posteriori probe residual in units of sigma_1 (0 when
 * no check ran) and how many fallbacks (Householder QR after a CholeskyQR breakdown, direct pass after a failed check) were taken. */
SB_API int sb_pca_diagnostics(sb_ctx *ctx, double *cond_r, double *probe_resid, int *fallbacks);
/* svd_rand (scan-rs/src/dim_red/rand_svd.rs:54-129); omega: (l x m) when n > m, (n_local x l) when m >= n */
SB_API int sb_randsvd(sb_nmat *a, uint32_t k, uint32_t l, uint32_t n_iter, uint64_t seed, const double *omega,
               double *U, double *S, double *V);
/* RandSvd::run_pca_cancellable (rand_svd.rs:44-49): l = max(k + 4, floor(k * l_multiplier)), seed 0 */
SB_API int sb_randsvd_run_pca(sb_nmat *a, uint32_t k, double l_multiplier, uint32_t n_iter, double *U, double *S,
                       double *V);

/* irlba (scan-rs/src/dim_red/irlba.rs:71-215): implicitly restarted Lanczos bidiagonalisation, nu triplets, tolerance tol
 * (Irlba::new: 1e-4), at most maxit restarts (50); working dimension m_b = min(nu + 20, 3 nu, n) (:87).  v0[n_local] = this rank's
 * slice of the start vector (normalised inside), or NULL for sb_irlba_start(0, n_global).  The reference draws it from rand_distr's
 * Normal on SmallRng seed 0, a third-party stream that cannot be restated offline (parity unpinned, like Omega).  The
 * `resid[i] < tol * smax` test carries no absolute value in the reference (:176-181); it is kept, with sign-canonical singular
 * vectors of the small matrix (largest-magnitude entry of each right vector positive).  Progress milestones it / maxit (:206).
 * Outputs U[m x nu], S[nu], V[n_local x nu] row-major; mprod_out / iters_out (optional): matrix products, restarts taken. */
SB_API int sb_irlba(sb_nmat *a, uint32_t nu, double tol, uint32_t maxit, const double *v0, sb_progress_cb cb, void *user,
             double *U, double *S, double *V, uint32_t *mprod_out, uint32_t *iters_out);
/* The builder-defined default start vector of sb_irlba: Box-Muller on the Xoshiro256++ stream of sb_omega, entry i for global cell i. */
SB_API int sb_irlba_start(uint64_t seed, uint64_t n, double *out);

/* ---------------------------------------------------------------- moment consumers (diff-exp's reads of the count matrix)
 * mean_var_axis (sqz/src/mat.rs:285-329): V[X] = E[X^2] - E[X]^2 along an axis.  axis 1: per gene over all cells (m values,
 * summed over ranks); axis 0: per local cell over the m genes.  cell_div (n_local values or NULL): the SizeNormalized view
 * `v as f64 / size_factor[c]` (diff-exp/src/diff_exp.rs:340-358; NaN factors become 0).  Without cell_div the sums are exact. */
SB_API int sb_mean_var_axis(sb_mat *mat, int axis, const double *cell_div, double *mean, double *var);
/* mean_var_rows (mat.rs:332-374): per gene over the listed cells (LOCAL indices of this rank's shard; a cell listed twice counts
 * twice, as the reference's CSC branch); the divisor is the number of listed cells over all ranks. */
SB_API int sb_mean_var_rows(sb_mat *mat, const uint64_t *cols, uint64_t n_cols, const double *cell_div, double *mean, double *var);
/* sum_rows / sum_cols / sum_rows_dual (mat.rs:414-476, 484-583) as exact u64 sums: per gene over the listed cells, per listed cell
 * over the genes, per gene over two lists at once (a cell in both lists adds to both). */
SB_API int sb_sum_rows(sb_mat *mat, const uint64_t *cols, uint64_t n_cols, uint64_t *out_m);
SB_API int sb_sum_cols(sb_mat *mat, const uint64_t *cols, uint64_t n_cols, uint64_t *out);
SB_API int sb_sum_rows_dual(sb_mat *mat, const uint64_t *cols1, uint64_t n1, const uint64_t *cols2, uint64_t n2, uint64_t *sum1,
                     uint64_t *sum2);
/* size_factors (diff_exp.rs:314-334): counts per cell / their median (50th percentile with linear interpolation,
 * diff-exp/src/stat.rs:107-163), over the listed local cells (NULL: all) of all ranks; umi_counts (optional) replaces the totals,
 * one value per listed cell.  out[n_local]: 0 at unlisted cells. */
SB_API int sb_size_factors(sb_mat *mat, const uint64_t *cells, uint64_t n_cells, const double *umi_counts, double *out);

/* ---------------------------------------------------------------- differential expression (diff-exp: sSeq, Cell Ranger's published test)
 * sb_sseq_compute_params replaces compute_sseq_params (diff-exp/src/diff_exp.rs; SURVEY 8f rank 4).  Over all N cells of all ranks:
 *   sf[c] = cell total / median of the totals (sb_size_factors); mean_g, var_g of the SizeNormalized view v / sf[c] (sb_mean_var_axis);
 *   use_g = var_g > 0;  S = sum_c 1 / sf[c];  phi_mm_g = max(0, (N var_g - mean_g S) / (mean_g^2 S)) on use_g, 0 elsewhere;
 *   zeta_hat = percentile of phi_mm_g[use_g] at zeta_quantile (rank q (n - 1), linear interpolation, the rule of the median);
 *   delta = (sum_use (phi_mm_g - mean(phi_mm[use]))^2 / (G - 1)) / (sum_use (phi_mm_g - zeta_hat)^2 / (G - 2)) with G = m (all genes);
 *   phi_g = (1 - delta) phi_mm_g + delta zeta_hat on use_g (0 there if no phi_mm_g[use_g] is > 0), NaN elsewhere.
 * SB_ERR_INVALID_ARG for a cell whose total is 0 and for a matrix without a gene of non-zero variance.
 * All arrays are caller-allocated; size_factors has n_local entries (this rank's cells), the gene arrays m (replicated). */
typedef struct sb_sseq_params {
    uint64_t num_cells;       /* N, over all ranks */
    uint32_t num_genes;       /* m */
    uint32_t reserved;
    double zeta_hat;
    double delta;
    double *size_factors;     /* [n_local] */
    double *gene_means;       /* [m] */
    double *gene_variances;   /* [m] */
    double *gene_moment_phi;  /* [m] phi_mm */
    double *gene_phi;         /* [m] shrunken dispersion */
    uint8_t *use_genes;       /* [m] 1 where var_g > 0 */
} sb_sseq_params;
/* The comparison-dependent results, each [n_comparisons x m] row-major, caller-allocated. */
typedef struct sb_diff_exp_out {
    uint64_t *sums_in;
    uint64_t *sums_out;
    double *normalized_mean_in;
    double *normalized_mean_out;
    double *p_values;
    double *adjusted_p_values;
    double *log2_fold_change;
} sb_diff_exp_out;
SB_API int sb_sseq_compute_params(sb_mat *mat, double zeta_quantile, sb_sseq_params *out);
/* sseq_differential_expression (diff_exp.rs): condition lists are strictly ascending LOCAL cell indices, each non-empty over all
 * ranks; params come from sb_sseq_compute_params (on sharded contexts: this rank's size factors, the replicated gene arrays).
 *   sums_in / sums_out: exact u64 sums over the listed cells; s_in / s_out = sum of sf over the listed cells (in global cell order);
 *   normalized_mean = sums / s;  log2_fold_change = log2((1 + sums_in) / (1 + s_in)) - log2((1 + sums_out) / (1 + s_out));
 *   p = 1 where use_g is 0.  With mu = mean_g, phi = phi_g:
 *   both sums > big_count (asymptotic): alpha = s_in mu / (1 + phi mu), beta = (s_out / s_in) alpha, T = x_in + x_out, med = median of
 *     Beta(alpha, beta); p = 2 I_{(x_in + 0.5) / T}(alpha, beta) if (x_in + 0.5) / T < med, else 2 (1 - I_{(x_in - 0.5) / T}(alpha, beta)),
 *     evaluated as 2 I_{1 - (x_in - 0.5) / T}(beta, alpha) (no cancellation); not clipped;
 *   otherwise (exact): lp(x, s) = lgamma(r + x) - (lgamma(r) + lgamma(x + 1)) + x log(mu s / (r + mu s)) + r log(r / (r + mu s)),
 *     r = s / phi (phi = 0: the Poisson limit -lgamma(x + 1) + x log(mu s) - mu s, builder-defined); l(x) = lp(x, s_in) + lp(T - x, s_out);
 *     p = exp(LSE_{x = 0..T, l(x) <= l(x_in)} l(x) - LSE_{x = 0..T} l(x)); bit-reproducible and independent of the rank count;
 *   adjusted_p_values: Benjamini-Hochberg over the use_g genes (q = min(1, cummin over descending p of p n / rank)), p elsewhere. */
SB_API int sb_sseq_diff_exp(sb_mat *mat, const sb_sseq_params *params, const uint64_t *cond_in, uint64_t n_in, const uint64_t *cond_out,
                     uint64_t n_out, uint64_t big_count, sb_diff_exp_out *out);
/* Cell Ranger's per-cluster loop, batched: comparison j is "labels == j" against "labels != j" (labels[n_local] of this rank's cells,
 * each < n_groups; n_groups >= 2; no group may be empty over all ranks).  out arrays are [n_groups x m]. */
SB_API int sb_sseq_one_vs_rest(sb_mat *mat, const sb_sseq_params *params, const uint32_t *labels, uint32_t n_groups, uint64_t big_count,
                        sb_diff_exp_out *out);
/* Pairwise comparisons of labelled groups, batched: comparison j is "labels == pairs[2j]" against "labels == pairs[2j + 1]"
 * (labels[n_local] of this rank's cells, each < n_groups; pairs[n_pairs x 2], n_pairs >= 1, each pair two different groups below
 * n_groups, neither empty over all ranks; else SB_ERR_INVALID_ARG).  One pass over the matrix for every pair; s of a group is its
 * cells' size factors summed in global cell order.  Every output row j equals sb_sseq_diff_exp called with the cells of the two
 * groups, bit for bit.  out arrays are [n_pairs x m]. */
SB_API int sb_sseq_pairs(sb_mat *mat, const sb_sseq_params *params, const uint32_t *labels, uint32_t n_groups, const uint32_t *pairs,
                  uint32_t n_pairs, uint64_t big_count, sb_diff_exp_out *out);

/* ---------------------------------------------------------------- kNN on the scores (next step of the pipeline)
 * knn / find_nn (scan-rs/src/nn.rs:38-83): for every query row (n_queries x dim, row-major) the indices of its k nearest points
 * (n_points x dim) in Euclidean distance, nearest first, into out[n_queries x k]; rows with fewer than k candidates are padded
 * with 0xFFFFFFFF (the reference pads with T::max_value(), nn.rs:67).  include_self = 0 skips the point with index
 * self_offset + row (knn() queries the tree with its own points; self_offset serves cell-sharded callers).  Among exactly
 * equidistant points the lower index comes first. */
SB_API int sb_knn(sb_ctx *ctx, const double *points, uint64_t n_points, uint32_t dim, const double *queries, uint64_t n_queries,
           uint32_t k, int include_self, uint64_t self_offset, uint32_t *out);

/* ---------------------------------------------------------------- graph clustering (the step between kNN and diff-exp)
 * Deterministic Louvain on a shared-nearest-neighbour graph; the base algorithm of the reference's `leiden` crate, made
 * synchronous so that the result is bit-reproducible and equal to oracle/louvain.py.
 *
 * sb_snn_graph: nbr[n x k] as sb_knn returns it (global indices, no self index, 0xFFFFFFFF only at row ends; 1 <= k <= 128,
 * n k < 2^28, else SB_ERR_UNSUPPORTED).  Edges {i, j} wherever j is in N(i) or i in N(j), stored both ways: indptr[n + 1],
 * columns ascending, no self loops.  Weight w = (s << 24) / u (integer division), s = |N+(i) n N+(j)|, u = |N+(i)| + |N+(j)| - s,
 * N+(i) = N(i) u {i}: the Jaccard index of the closed neighbourhoods in 24-bit fixed point.  indices / weights must hold 2 n k
 * entries; *nnz receives the count.  An index >= n, a self index, a duplicate in a row or padding before a row end is
 * SB_ERR_INVALID_ARG.
 *
 * sb_louvain: a host CSR of n nodes, symmetric (equal weights both ways), no duplicate entry, self loops allowed (checked on the
 * device: SB_ERR_INVALID_ARG); 2m = sum of all entries must be < 2^53 (SB_ERR_UNSUPPORTED).  K_i = row sum (a self loop once),
 * S_c = sum of K over c, e_ic = weight from i to the members of c other than i.  Level: every node starts alone; iteration t moves
 * every node i (community a) to the allowed neighbouring c with the largest
 *   gain(c) = ((double)e_ic - (double)e_ia) - g2m (double)K_i ((double)S_c - (double)(S_a - K_i)),  g2m = resolution / (double)2m,
 * evaluated in this order without contraction, if that gain is > 0 (ties: the smallest c).  Allowed: c > a in even iterations,
 * c < a in odd ones.  The moves are kept only if Q = (double)sum_I / (double)2m - resolution sum_S2 / (2m)^2 strictly increases
 * (sum_I: intra-community directed weight, self loops included; sum_S2 = sum S_c^2 exact in 128 bits, as (double)hi 2^64 +
 * (double)lo).  A level ends after two consecutive iterations without a kept move, or max_iterations.  A level that kept a move
 * is aggregated (communities numbered in ascending id; coarse weights summed per pair, self loops carrying the internal weight)
 * and the next level runs, up to max_levels.  Labels: clusters numbered by size, descending, ties to the smallest node index
 * (0..n_clusters-1, none empty).  A graph of total weight 0 leaves every node its own cluster (one level, 0 iterations, Q = 0).
 *
 * sb_cluster_knn: sb_snn_graph + sb_louvain with the graph kept on the device.  On a cell-sharded context every rank passes its own
 * rows (n_local x k, global indices: sb_knn with self_offset = its first cell) and receives its cells' labels; the rows are
 * gathered in global cell order and every rank runs the same clustering, so labels equal world 1 bit for bit. */
#define SB_LOUVAIN_MAX_LEVELS 32
typedef struct sb_louvain_opts {
    double resolution;        /* gamma > 0 (default 1.0) */
    uint32_t max_levels;      /* 1..SB_LOUVAIN_MAX_LEVELS (default 32) */
    uint32_t max_iterations;  /* per level, >= 1 (default 100) */
} sb_louvain_opts;            /* NULL: the defaults */
typedef struct sb_louvain_info {
    uint32_t n_clusters;
    uint32_t n_levels;
    double modularity;        /* Q of the final partition */
    uint64_t level_nodes[SB_LOUVAIN_MAX_LEVELS];
    uint32_t level_iterations[SB_LOUVAIN_MAX_LEVELS];
    double level_modularity[SB_LOUVAIN_MAX_LEVELS];
} sb_louvain_info;
SB_API int sb_snn_graph(sb_ctx *ctx, const uint32_t *nbr, uint64_t n, uint32_t k, uint64_t *indptr, uint32_t *indices, uint64_t *weights,
                 uint64_t *nnz);
SB_API int sb_louvain(sb_ctx *ctx, uint64_t n, const uint64_t *indptr, const uint32_t *indices, const uint64_t *weights,
               const sb_louvain_opts *opts, uint32_t *labels, sb_louvain_info *info);
SB_API int sb_cluster_knn(sb_ctx *ctx, const uint32_t *nbr, uint64_t n_local, uint32_t k, const sb_louvain_opts *opts, uint32_t *labels,
                   sb_louvain_info *info);

/* ---------------------------------------------------------------- merging of over-split clusters (Cell Ranger's MERGE_CLUSTERS)
 * scan-rs's linkage.rs and merge_clusters.rs, restated (neither is pinned here); oracle/merge_clusters.py restates the rule literally.
 *
 * sb_linkage_complete: host only, no context.  points[n x dim] (f64, row-major, finite; else SB_ERR_INVALID_ARG), 1 <= n <= 4,096
 * (SB_ERR_UNSUPPORTED above), dim >= 1 -> Z[(n - 1) x 4] in scipy's layout (scipy.cluster.hierarchy.linkage(method="complete")).
 *   d(i, j) = sqrt(sum_c (x_j,c - x_i,c)^2), summed in coordinate order without contraction (knn.cu's expression); a non-finite
 *   distance is SB_ERR_INVALID_ARG.  Between clusters the largest point distance.  NN-chain: the chain starts at the lowest active
 *   slot; its next element is the active slot nearest to the top -- on a tie the element below the top wins, otherwise the lowest
 *   slot; two mutual nearest neighbours x < y merge at height d(x, y) into slot y.  The merges are stably sorted by height (equal
 *   heights keep merge order) and numbered as scipy does: row i = (id_a < id_b, height, size), the new cluster is id n + i.
 *
 * sb_merge_clusters: labels[n_local] (each < n_groups, no group empty over all ranks, 1 <= n_groups <= 4,096: SB_ERR_UNSUPPORTED
 * above), scores[n_local x dim] (the PCA scores, finite, 1 <= dim <= 128), params from sb_sseq_compute_params on the whole matrix.
 * Each round, with the current clusters numbered 0..K-1 in ascending id:
 *   1. centroid of a cluster: every score column summed over its cells in ascending global cell order (one rounding per add),
 *      divided by the cell count;
 *   2. Z = sb_linkage_complete of the centroids;
 *   3. candidates: every row of Z whose two children are both leaves (< K); they are disjoint;
 *   4. one batched pairwise sSeq test (sb_sseq_pairs' path) of every candidate (a, b), a < b, the lower id as the in-group;
 *   5. a pair merges when fewer than min_de_genes genes have adjusted p < adj_p_threshold; the merged cluster keeps id a;
 *   6. the survivors are renumbered 0..K'-1 in ascending old id.
 * Rounds repeat until one merges nothing or one cluster is left (n_rounds counts the rounds that tested pairs).  labels_out[n_local]:
 * the final clusters numbered by size, descending, ties to the smallest global cell index (sb_cluster_knn's rule, so labels no round
 * merges come back unchanged).  On a cell-sharded context every rank passes its own labels, score rows and params and receives its
 * cells' labels; labels, size factors and scores are gathered in global cell order, so the result equals world 1 bit for bit. */
#define SB_LINKAGE_MAX_POINTS 4096
typedef struct sb_merge_opts {
    double adj_p_threshold;  /* 0 < t <= 1 (default 0.05) */
    uint32_t min_de_genes;   /* a pair with fewer DE genes merges (default 1) */
    uint32_t reserved;       /* 0 */
    uint64_t big_count;      /* sSeq's switch to the asymptotic test (default 900) */
} sb_merge_opts;             /* NULL: the defaults */
typedef struct sb_merge_info {
    uint32_t n_clusters;
    uint32_t n_rounds;
    uint64_t pairs_tested;
    uint64_t pairs_merged;
} sb_merge_info;
SB_API int sb_linkage_complete(const double *points, uint32_t n, uint32_t dim, double *Z);
SB_API int sb_merge_clusters(sb_mat *mat, const sb_sseq_params *params, const double *scores, uint32_t dim, const uint32_t *labels,
                      uint32_t n_groups, const sb_merge_opts *opts, uint32_t *labels_out, sb_merge_info *info);

/* ---------------------------------------------------------------- UMAP embedding (the reference's `umap-rs`, a port of umap-learn)
 * The fuzzy kNN graph and umap-learn's layout, made epoch-synchronous so that the result is bit-reproducible at every grid and
 * world size; restated by oracle/umap.py.
 *
 * sb_umap_graph: scores X[n x dim] (f64, row-major; the PCA scores) and nbr[n x k] as sb_knn(..., include_self = 0) returns them
 * (1 <= k <= 128, n k < 2^28, else SB_ERR_UNSUPPORTED; an index >= n, a self index, a duplicate in a row or padding before a row
 * end is SB_ERR_INVALID_ARG).  umap-learn's n_neighbors is k + 1 (the point itself at distance 0).
 *   d_ij  = sqrt(sum_c (x_j,c - x_i,c)^2), summed in coordinate order without contraction (knn.cu's ranking expression);
 *   rho_i = the smallest non-zero d_ij of the row (0 if none);
 *   sigma_i by umap-learn's smooth_knn_dist bisection: lo = 0, hi = inf, mid = 1; 64 steps of psum = sum over the listed j, in
 *           slot order, of (d_ij - rho_i > 0 ? exp(-((d_ij - rho_i) / mid)) : 1); stop when |psum - log2(k + 1)| < 1e-5; psum >
 *           target: hi = mid, mid = (lo + hi) / 2; else lo = mid, mid = hi == inf ? 2 mid : (lo + hi) / 2.  Floors: sigma_i >=
 *           1e-3 (s_i / (m_i + 1)) when rho_i > 0, else >= 1e-3 (sum_i s_i / sum_i (m_i + 1)); s_i = the row's distances summed
 *           in slot order, m_i = its listed count, the rows summed in order;
 *   w_ij  = exp(-max(0, d_ij - rho_i) / sigma_i);
 *   union = mix ((a + b) - a b) + (1 - mix) (a b), a = w_ij, b = w_ji (0 when not listed), mix = set_op_mix_ratio; stored both
 *           ways, columns ascending, no self loops, zero weights dropped.
 * indices / weights must hold 2 n k entries; *nnz receives the count; rho / sigma (n each) may be NULL.
 *
 * sb_umap_layout: a host CSR of n vertices, symmetric (equal weights both ways), no duplicate entry, weights in (0, 1] (checked
 * on the device: SB_ERR_INVALID_ARG); a row's entries are taken with columns ascending.  Schedule (umap-learn's
 * optimize_layout_euclidean, arithmetic in f64): n_epochs (0: 500 if n <= 10,000 else 200); entries with w < w_max / n_epochs
 * dropped; per remaining directed entry e (in CSR order) eps = w_max / w, epn = eps / negative_sample_rate, next = eps,
 * next_neg = epn.  Epoch t = 0..n_epochs-1, alpha = learning_rate (1 - t / n_epochs), reads one snapshot Y of the positions; every
 * entry (head j, tail k) with next <= t:
 *   attractive: d2 = |y_j - y_k|^2 (coordinate order); g = d2 > 0 ? ((-2 a) b) d2^(b - 1) / (a d2^b + 1) : 0; per coordinate
 *               c = alpha clip(g (y_j - y_k)) goes to j and -c to k;
 *   next += eps; s = max(0, trunc((t - next_neg) / epn)) negative samples, the p-th one v = mix64(mix64(mix64(mix64(seed) ^ t)
 *               ^ e) ^ p) % n (mix64: SplitMix64's finaliser; e: the entry's index after pruning); v = j is skipped; d2 > 0:
 *               c = alpha clip((2 gamma b) / ((0.001 + d2) (a d2^b + 1)) (y_j - y_v)), d2 = 0: c = 4 alpha, to j;
 *               next_neg += s epn.
 * clip(x) = max(-4, min(4, x)).  Every contribution is rounded to an integer q = rint(c 2^32), summed per vertex in 64 bits and
 * added once at the end of the epoch; positions are those integers (y = q 2^-32), so the layout does not depend on the order of
 * the sums.  A graph whose largest degree could let an epoch's sum pass 2^62 is SB_ERR_UNSUPPORTED.  (a, b): given (both > 0),
 * or fitted: 1 / (1 + a x^(2b)) to umap-learn's target (1 for x < min_dist, exp(-(x - min_dist) / spread) beyond) on
 * linspace(0, 3 spread, 300) by Levenberg-Marquardt from (1, 1).  Start (init[n x n_components], f64): SB_UMAP_INIT_PCA scales
 * every column to [0, 10] as 10 (x - min) / (max - min) (a constant column: 0), SB_UMAP_INIT_USER takes it as given (finite,
 * |x| < 2^30), SB_UMAP_INIT_RANDOM ignores it: uniform [-10, 10) as -10 + 20 ((h >> 11) 2^-53), h = mix64(mix64(mix64(seed)
 * ^ (2^64 - 1)) ^ (i n_components + c)).  Either start is rounded to multiples of 2^-32.  out[n x n_components] (f64).
 *
 * sb_umap: sb_umap_graph + sb_umap_layout with the graph kept on the device; SB_UMAP_INIT_PCA starts from the first n_components
 * columns of X, SB_UMAP_INIT_USER from init (this rank's rows).  On a cell-sharded context every rank passes its own rows of X
 * and nbr (global indices: sb_knn with self_offset = its first cell) and receives its own rows of the embedding; the rows are
 * gathered in global cell order and every rank runs the same layout, so the embedding equals world 1 bit for bit. */
#define SB_UMAP_INIT_PCA 0
#define SB_UMAP_INIT_RANDOM 1
#define SB_UMAP_INIT_USER 2
typedef struct sb_umap_opts {
    uint32_t n_components;          /* 1..8 (default 2) */
    uint32_t n_epochs;              /* 0: 500 if n <= 10,000, else 200 (default 0) */
    double min_dist;                /* 0 <= min_dist <= spread (default 0.1) */
    double spread;                  /* > 0 (default 1.0) */
    double a, b;                    /* both 0: fitted from min_dist / spread (default); both > 0: used as given */
    double learning_rate;           /* > 0 (default 1.0) */
    double repulsion_strength;      /* gamma >= 0 (default 1.0) */
    double set_op_mix_ratio;        /* 0..1 (default 1.0: fuzzy union; 0: fuzzy intersection) */
    uint32_t negative_sample_rate;  /* negative samples per positive sample (default 5) */
    uint32_t init;                  /* SB_UMAP_INIT_PCA (default), SB_UMAP_INIT_RANDOM, SB_UMAP_INIT_USER */
    uint64_t seed;                  /* negative samples and the random start (default 0) */
} sb_umap_opts;                     /* NULL: the defaults */
typedef struct sb_umap_info {
    double a, b;                    /* as used */
    double max_weight;              /* w_max of the graph */
    uint64_t n_edges;               /* directed entries of the graph */
    uint64_t n_edges_used;          /* after pruning */
    uint32_t n_epochs;
} sb_umap_info;
SB_API int sb_umap_graph(sb_ctx *ctx, const double *scores, const uint32_t *nbr, uint64_t n, uint32_t dim, uint32_t k, const sb_umap_opts *opts,
                  uint64_t *indptr, uint32_t *indices, double *weights, uint64_t *nnz, double *rho, double *sigma);
SB_API int sb_umap_layout(sb_ctx *ctx, uint64_t n, const uint64_t *indptr, const uint32_t *indices, const double *weights, const double *init,
                   const sb_umap_opts *opts, double *out, sb_umap_info *info);
SB_API int sb_umap(sb_ctx *ctx, const double *scores, const uint32_t *nbr, uint64_t n_local, uint32_t dim, uint32_t k, const sb_umap_opts *opts,
            const double *init, double *out, sb_umap_info *info);

/* ---------------------------------------------------------------- t-SNE embedding (the reference's `bhtsne`, van der Maaten's
 * Barnes-Hut t-SNE) with bhtsne's parameter names, defaults and schedule; restated by oracle/tsne.py.
 *
 * Ordered sums: a sum over m values is taken in chunks of 1,024 (chunk c: values [1024 c, 1024 (c + 1))), each chunk left to right
 * from its first value, then the chunk sums left to right.  The order depends on m alone, never on the grid, the SM count or the
 * world size.
 *
 * sb_tsne_affinities: scores X[n x dim] (f64, row-major) and nbr[n x k] as sb_knn(..., include_self = 0) returns them.  bhtsne
 * lists K = floor(3 perplexity) neighbours: callers pass k = min(n - 1, K).  SB_ERR_INVALID_ARG: perplexity not finite or not > 0,
 * n - 1 < 3 perplexity, k < min(n - 1, K), an index >= n, a self index, a duplicate in a row, padding before a row end;
 * SB_ERR_UNSUPPORTED: k > 128, n k >= 2^28.  All listed slots of a row are used.
 *   scaling  X minus its column means (ordered sums over the cells, / n), then divided by the largest |x| (skipped when 0), as
 *            bhtsne's run does;
 *   d_ij     sqrt(sum_c (x_j,c - x_i,c)^2) in coordinate order without contraction (knn.cu's ranking expression); D_ij = d_ij d_ij;
 *   beta_i   bhtsne's computeGaussianPerplexity: beta = 1, min = -DBL_MAX, max = DBL_MAX; at most 200 steps of p_j = exp(-(beta D_ij)),
 *            sum_P = DBL_MIN + the p_j in slot order, H = (sum over slots of beta (D_ij p_j)) / sum_P + log(sum_P); stop when
 *            |H - log(perplexity)| < 1e-5; H above: min = beta, beta = max still +-DBL_MAX ? 2 beta : (beta + max) / 2; below:
 *            max = beta, beta = min still +-DBL_MAX ? beta / 2 : (beta + min) / 2.  P_j|i = p_j / sum_P of the last step; beta[i]
 *            is the beta of that step;
 *   P        P_ij = P_j|i + P_i|j (0 when not listed), zeros dropped, stored both ways with columns ascending, then divided by
 *            their total (an ordered sum in CSR order).
 * indices / P must hold 2 n k entries; *nnz receives the count; beta (n) may be NULL.
 *
 * sb_tsne_layout: P as a host CSR of n points: symmetric (equal values both ways), no duplicate entry, entries in (0, 1] (checked
 * on the device: SB_ERR_INVALID_ARG); a row is taken with columns ascending.  n_components must be 2 (else SB_ERR_UNSUPPORTED).
 * Start (init[n x 2], f64): SB_TSNE_INIT_PCA (default) takes the two columns divided by the population standard deviation of
 * column 0 (ordered sums: the mean, then the squared deviations; a zero or non-finite deviation is SB_ERR_INVALID_ARG) times 1e-4,
 * as sklearn and openTSNE do; SB_TSNE_INIT_USER takes them as given (finite); SB_TSNE_INIT_RANDOM ignores them: point i gets
 * 1e-4 (r cos a, r sin a), r = sqrt(-2 log u1), a = 6.283185307179586 u2, u1 = ((h(2i) >> 11) + 1) 2^-53, u2 = (h(2i + 1) >> 11)
 * 2^-53, h(x) = mix64(mix64(mix64(seed) ^ (2^64 - 1)) ^ x) (mix64: SplitMix64's finaliser), bhtsne's N(0, 1e-4^2).
 * Iteration t = 0..max_iter-1 (no host round trip inside the loop; every operation below is one correctly rounded f64 op):
 *   tree     root box: centre = the mean of Y (ordered sums / n), half-width h_a = max(max_a - mean_a, mean_a - min_a) + 1e-5;
 *            per point and axis q_a = floor((y_a - (mean_a - h_a)) / (h_a + h_a) 2^32) clamped to [0, 2^32 - 1]; the 64-bit Morton
 *            code has the bits of q_x at the odd positions (bit 63 the top x bit) and of q_y at the even.  Codes sorted (ties in
 *            cell order); a run of equal codes is one leaf; the internal nodes are the binary radix tree of the distinct codes
 *            (Karras 2012).  A leaf's count and sum of y are its run summed in sorted order; an internal node's are left + right.
 *            An internal node with a common prefix of p bits has half-widths h_x 2^-ceil(p/2), h_y 2^-floor(p/2).
 *   forces   for every point i: pos_i = sum over its CSR row (columns ascending) of ((e P_ij) / ((1 + b_x b_x) + b_y b_y)) b,
 *            b = y_i - y_j, e = early_exaggeration for t <= stop_lying_iter, else 1.  neg_i and q_i: a walk from the root, left
 *            child before right; a node's centre c = sum / count (a leaf holding i: count - 1 points at (sum - y_i) / (count - 1),
 *            skipped when count = 1), b = y_i - c, D = b_x b_x + b_y b_y; an internal node is opened unless max(half-widths) / sqrt(D)
 *            < theta; otherwise (and at every leaf) w = 1 / (1 + D), q_i += count w, neg_i += ((count w) w) b.  theta = 0 gives the
 *            exact gradient.  sum_Q = the ordered sum of q_i over the points in cell order.
 *   update   dY = pos - neg / sum_Q; gains (from 1): sign(dY) != sign(uY) ? gains + 0.2 : gains 0.8, floor 0.01; uY (from 0) =
 *            mom uY - (eta gains) dY, mom = 0.5 for t <= mom_switch_iter, else 0.8; Y += uY; then Y minus its mean (ordered sums).
 * eta = learning_rate, or max(n / (4 early_exaggeration), 50) when it is 0.  info: kl_divergence as bhtsne's evaluateError
 * estimates it on the final Y (sum_Q from the same walk; sum of P_ij log((P_ij + FLT_MIN) / (Q_ij + FLT_MIN)), Q_ij = (1 / (1 +
 * |y_i - y_j|^2)) / sum_Q, per row in CSR order, the rows in an ordered sum), the learning rate used, the entries of P and the
 * iterations.  out[n x 2] (f64).
 *
 * sb_tsne: sb_tsne_affinities + sb_tsne_layout with P kept on the device; SB_TSNE_INIT_PCA starts from the first two columns of the
 * (unscaled) scores, SB_TSNE_INIT_USER from init (this rank's rows).  On a cell-sharded context every rank passes its own rows of X
 * and nbr (global indices) and receives its own rows of the embedding; the rows are gathered in global cell order and every rank
 * runs the same layout, so the embedding equals world 1 bit for bit.
 * Parity with the `bhtsne` crate is not pinned: its source is not part of this project. */
#define SB_TSNE_INIT_PCA 0
#define SB_TSNE_INIT_RANDOM 1
#define SB_TSNE_INIT_USER 2
typedef struct sb_tsne_opts {
    double perplexity;          /* > 0 (default 30) */
    double theta;               /* Barnes-Hut accuracy, >= 0 (default 0.5; 0: exact) */
    double learning_rate;       /* eta >= 0 (default 200; 0: max(n / (4 early_exaggeration), 50)) */
    double early_exaggeration;  /* > 0 (default 12) */
    uint32_t max_iter;          /* iterations (default 1000) */
    uint32_t stop_lying_iter;   /* last iteration with the exaggeration (default 250) */
    uint32_t mom_switch_iter;   /* last iteration with momentum 0.5 (default 250) */
    uint32_t n_components;      /* 2 */
    uint32_t init;              /* SB_TSNE_INIT_PCA (default), SB_TSNE_INIT_RANDOM, SB_TSNE_INIT_USER */
    uint32_t reserved;          /* 0 */
    uint64_t seed;              /* the random start (default 0) */
} sb_tsne_opts;                 /* NULL: the defaults */
typedef struct sb_tsne_info {
    double kl_divergence;       /* bhtsne's estimate on the final embedding */
    double learning_rate;       /* as used */
    uint64_t nnz;               /* entries of P */
    uint32_t n_iter;
    uint32_t reserved;
} sb_tsne_info;
SB_API int sb_tsne_affinities(sb_ctx *ctx, const double *scores, const uint32_t *nbr, uint64_t n, uint32_t dim, uint32_t k, const sb_tsne_opts *opts,
                       uint64_t *indptr, uint32_t *indices, double *P, uint64_t *nnz, double *beta);
SB_API int sb_tsne_layout(sb_ctx *ctx, uint64_t n, const uint64_t *indptr, const uint32_t *indices, const double *P, const double *init,
                   const sb_tsne_opts *opts, double *out, sb_tsne_info *info);
SB_API int sb_tsne(sb_ctx *ctx, const double *scores, const uint32_t *nbr, uint64_t n_local, uint32_t dim, uint32_t k, const sb_tsne_opts *opts,
            const double *init, double *out, sb_tsne_info *info);

/* ---------------------------------------------------------------- measurement
 * Device-side timing on the context's own stream (CUDA events) and per-kernel accounting;
 * bench.py builds its roofline object from these.  Not part of the reference interface. */
typedef struct {
    double spmm_t_ms;     /* K7: out[cells x w]  = A^T . Y  (cell-major gather) */
    double spmm_n_ms;     /* K8: out[genes x w]  = A . X    (gene-major panel gather) */
    double moments_ms;    /* K5 */
    double reduce_ms;     /* integer reductions K1/K2 */
    double dense_ms;      /* QR / Gram / eigh / small GEMMs */
    double comm_ms;       /* NCCL collectives */
    double spmm_t_bytes;  /* algorithmic bytes summed over launches (SURVEY 8d formula) */
    double spmm_n_bytes;
    double spmm_t_flops;
    double spmm_n_flops;
    uint64_t spmm_t_launches;
    uint64_t spmm_n_launches;
    uint64_t kernel_launches; /* every kernel this library launched (own + library calls) */
    uint64_t own_kernel_launches;
    double upload_ms;     /* sb_upload: host -> device copies */
    double build_ms;      /* sb_upload: device-side layout build (sorts, dense panel) */
    double output_ms;     /* device -> host copies of U, sigma, V */
} sb_profile;
SB_API int sb_profile_enable(sb_ctx *ctx, int on); /* on: record a CUDA-event pair around every phase */
SB_API int sb_profile_reset(sb_ctx *ctx);
SB_API int sb_profile_get(sb_ctx *ctx, sb_profile *out);
SB_API int sb_timer_begin(sb_ctx *ctx);            /* records an event on the context stream */
SB_API int sb_timer_end(sb_ctx *ctx, float *ms);   /* records, synchronises, returns elapsed ms */
/* write >= 2x L2 worth of bytes so the next timed step starts cold */
SB_API int sb_flush_l2(sb_ctx *ctx);

/* ---------------------------------------------------------------- synthetic workload
 * Test/bench utility, not part of the reference interface: negative-binomial count matrix
 * from a counter-based hash keyed by (seed, gene, global cell), identical bit for bit to
 * the CPU generator in synth/ (see synth_nb.h).  pf[n_clusters x m] are per-cluster gene
 * abundances, depth[n_local] per-cell depths, cluster[n_local] cluster ids. */
SB_API int sb_synth_generate(sb_ctx *ctx, uint32_t m, uint64_t n_local, uint64_t cell_offset, uint64_t seed,
                      uint32_t n_clusters, const double *pf, const double *depth, const uint8_t *cluster,
                      uint32_t r_dispersion, sb_mat **out);

#ifdef __cplusplus
}
#endif
#endif /* SCANB200_H */
