// common.cuh -- internal structures of libscanb200 (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <cublas_v2.h>
#include <cusolverDn.h>
#include "nccl_shim.h"

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/scanb200.h"
#include "gather_units.h"  // GUnit + the host-side cutting of the gather streams into work units

typedef uint32_t u32;
typedef uint64_t u64;

// ---------------------------------------------------------------- errors
void sb_set_error(const char *fmt, ...);
int sb_fail(int code, const char *fmt, ...);

#define SB_CUDA(expr)                                                                         \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return sb_fail(_e == cudaErrorMemoryAllocation ? SB_ERR_OOM : SB_ERR_CUDA,        \
                           "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__,      \
                           __LINE__, cudaGetErrorString(_e));                                 \
    } while (0)
#define SB_CUBLAS(expr)                                                                       \
    do {                                                                                      \
        cublasStatus_t _s = (expr);                                                           \
        if (_s != CUBLAS_STATUS_SUCCESS)                                                      \
            return sb_fail(SB_ERR_LINALG, "cuBLAS error %d at %s:%d", (int)_s, __FILE__, __LINE__); \
    } while (0)
#define SB_CUSOLVER(expr)                                                                     \
    do {                                                                                      \
        cusolverStatus_t _s = (expr);                                                         \
        if (_s != CUSOLVER_STATUS_SUCCESS)                                                    \
            return sb_fail(SB_ERR_LINALG, "cuSOLVER error %d at %s:%d", (int)_s, __FILE__, __LINE__); \
    } while (0)
#define SB_NCCL(expr)                                                                         \
    do {                                                                                      \
        ncclResult_t _r = (expr);                                                             \
        if (_r != ncclSuccess)                                                                \
            return sb_fail(SB_ERR_NCCL, "NCCL error %s at %s:%d", ncclGetErrorString(_r),     \
                           __FILE__, __LINE__);                                               \
    } while (0)
#define SB_TRY(expr)                 \
    do {                             \
        int _rc = (expr);            \
        if (_rc != SB_OK) return _rc; \
    } while (0)

// ---------------------------------------------------------------- device buffer (RAII)
// Stream-ordered allocations from the device's default memory pool (release threshold raised to
// "never" in sb_init), so the dozens of temporaries per PCA call cost microseconds instead of a
// cudaMalloc/cudaFree device synchronisation each.  The stream is the calling context's stream,
// published by every API entry through sb_set_alloc_stream().
cudaStream_t sb_alloc_stream();
cudaMemPool_t sb_alloc_pool();
void sb_set_alloc_stream(cudaStream_t s, cudaMemPool_t pool = nullptr);
// streams of live contexts: a buffer that outlives its context (a handle freed after sb_shutdown) is returned with a plain cudaFree
bool sb_stream_alive(cudaStream_t s);
// Exact-size block cache in front of the context's memory pool (ctx.cu).  A call sequence that repeats (upload -> normalize -> PCA
// -> free, per data set) asks for the same large sizes in the same order; handing a freed block straight to the next request of
// that size keeps the pool's free list out of it -- the pool otherwise re-stitches physical memory into new virtual ranges
// whenever its free blocks do not fit (measured: +13 ms of compute and +15 ms of upload per end-to-end step after the staging
// buffers changed size).  Same ordering contract as cudaFreeAsync / cudaMallocAsync on the context's stream.
void *sb_cache_take(cudaStream_t st, size_t bytes);
bool sb_cache_give(cudaStream_t st, void *p, size_t bytes);
void sb_cache_flush(cudaStream_t st);
void sb_cache_configure(cudaStream_t st, size_t cap_bytes);
#define SB_CACHE_MIN_BYTES ((size_t)1 << 20)
void sb_stream_register(cudaStream_t s, bool alive);

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaStream_t st = nullptr;
    DevBuf() {}
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    void release() {
        // a buffer that outlives its context (a handle freed after sb_shutdown) needs no free: its memory went with the context's pool
        if (p && sb_stream_alive(st)) {
            const size_t bytes = (n ? n : 1) * sizeof(T);
            if (bytes < SB_CACHE_MIN_BYTES || !sb_cache_give(st, p, bytes)) cudaFreeAsync(p, st);
        }
        p = nullptr;
        n = 0;
    }
    int alloc(size_t count) {
        release();
        n = count;
        if (count == 0) count = 1;
        st = sb_alloc_stream();
        if (count * sizeof(T) >= SB_CACHE_MIN_BYTES) {
            p = static_cast<T *>(sb_cache_take(st, count * sizeof(T)));
            if (p) return SB_OK;
        }
        cudaMemPool_t pool = sb_alloc_pool();
        cudaError_t e = pool ? cudaMallocFromPoolAsync((void **)&p, count * sizeof(T), pool, st) : cudaMallocAsync((void **)&p, count * sizeof(T), st);
        if (e == cudaErrorMemoryAllocation) {  // the cache may be sitting on the memory: give it back to the pool and ask again
            cudaGetLastError();
            sb_cache_flush(st);
            e = pool ? cudaMallocFromPoolAsync((void **)&p, count * sizeof(T), pool, st) : cudaMallocAsync((void **)&p, count * sizeof(T), st);
        }
        if (e != cudaSuccess) {
            p = nullptr;
            n = 0;
            cudaGetLastError();
            return sb_fail(e == cudaErrorMemoryAllocation ? SB_ERR_OOM : SB_ERR_CUDA,
                           "cudaMallocAsync of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
        }
        return SB_OK;
    }
    int ensure(size_t count) { return count <= n && p ? SB_OK : alloc(count); }
    void swap(DevBuf &o) {
        T *tp = p; p = o.p; o.p = tp;
        size_t tn = n; n = o.n; o.n = tn;
        cudaStream_t ts = st; st = o.st; o.st = ts;
    }
};

// ---------------------------------------------------------------- profile phases
enum Phase { PH_SPMM_T = 0, PH_SPMM_N, PH_MOMENTS, PH_REDUCE, PH_DENSE, PH_COMM, PH_UPLOAD, PH_BUILD, PH_OUTPUT, PH_COUNT };

struct sb_ctx {
    int device = 0;
    int sm_count = 148;
    size_t l2_bytes = 0;
    cudaStream_t stream = nullptr;
    cudaMemPool_t pool = nullptr;        // the context's own stream-ordered memory pool (nothing is changed on the device's default pool)
    cudaStream_t copy_stream = nullptr;  // host -> device copies of the pipelined upload
    cudaStream_t aux_stream = nullptr;   // the dense panel kernels when overlapped with the sparse kernels
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // Experimental (default off, measured slower -- DESIGN.md 3): run the sparse and the DMMA panel kernel of a product on two
    // streams with CTAs of both resident on every SM.
    bool overlap = false;    // A.X
    bool overlap_t = false;  // A^T.Y
    cublasHandle_t cublas = nullptr;
    cusolverDnHandle_t cusolver = nullptr;
    ncclComm_t comm = nullptr;
    int nranks = 1, rank = 0;
    int dense_cap = 2048;            // max genes in the dense hot panel (0 disables the hybrid layout)
    double dense_min_density = 0.12; // a gene joins the panel only if nnz/n_global is at least this
    bool panel_i8 = false;           // EXPERIMENTAL (panel_i8.cu): T-side dense panel on tcgen05 int8 instead of FP64 mma.sync
    int dense_max_count = 15;        // largest count kept in the dense panel of matrices uploaded afterwards (<= 15)
    // dense half of the hybrid layout of matrices built afterwards: 0 none, 1 u8 panel on the FP64 mma.sync path (dense_panel.cu),
    // 2 bit planes on the int8 tensor cores (planes.cu)
    int panel_mode = 2;
    int pl_debug = 0;                // timing experiments only (planes.cu): 1 no output reductions, 2 no epilogue arithmetic, 4 no tile expansion
    int pl_variant = 3;              // kernel generations of planes.cu (A/B): bit 0 T side (warp layout, paired stages), bit 1 N side (bulk-copied digit rows, 12 producers)
    int plane_items_per_cta = 48;    // T-side plane kernel: work items per CTA on its queue (tail length vs boundary cost)
    int plane_cap = 12288;           // most ranks a plane may cover
    int plane_levels = 6;            // most count levels kept as planes (<= PL_MAX_LEVELS)
    double plane_min_density = 0.01; // a 128-rank block joins level k only if this fraction of the cells has exactly that count
    bool gemm_skinny = true;         // tall products with at most 16 output columns: row-per-thread kernel instead of the 128-column MMA tiles
    bool eig_host = true;            // Gram matrices of order <= 128: k largest eigenpairs on the host (eig_host.h) instead of cuSOLVER syevd
    void *eig_pinned = nullptr;      // page-locked staging of that round trip
    size_t eig_pinned_bytes = 0;
    int eig_host_declined = 0;       // times the host solver's own check sent a matrix to the library solver
    int upload_chunks = 8;           // pipelined upload: chunks of whole cell blocks in flight between the copy engine and the layout build
    bool upload_sync = true;         // pipelined upload: synchronise the build stream after every chunk (matrix.cu)
    bool gather_defer = true;        // T-side gather under the plane kernels: run factor L_c(1) applied by k_pl_reduce_t instead of at every run end
    int gather_calibrate = 1;        // T-side gather: number of timed passes (per matrix) after which the static shares are re-cut by the measured panel rates (0 = off)
    double gather_seg_cost = 0.0;    // T-side gather cost model: fixed cost of a non-empty (cell block, gene panel) segment, in entries
    double gather_flush_cost = 5.0;  // T-side gather cost model: cost of a run end (flush: ~25 instructions + 20 reductions) in entries
    int gather_items_per_cta = 1;    // T-side gather: work items per CTA on the ticket queue (1 = one static share per CTA; 6 measured slower: 7.28 vs 6.85 ms per C3 pass -- finer pieces re-stage panels and lose the L2 locality of sweeping the cell blocks together)
    bool use_gather = true;          // panelled gather kernels (gather.cu); false: the first-generation K7 / K8 of spmm.cu
    bool direct_projection = false;  // true: always run the wide Q^T A pass (bk_svd.rs:102,131) instead of the R^-T identity
    bool verify_projection = false;  // true: always check the R^-T identity a posteriori (default: only when cond(R) > 1e9)
    bool eig_jacobi = false;         // 1: cusolverDnDsyevj for Gram matrices of order <= 192 (measured 2.7 ms vs syevd 1.8 + its ~230 launches at w = 100: no gain)
    bool own_dense = true;           // QR / Gram / projections on the repo's kernels (dense_own.cu); false: cuSOLVER / cuBLAS (dense.cu)
    double last_cond_r = 0.0, last_probe_resid = 0.0;  // diagnostics of the last sb_bksvd
    int last_fallbacks = 0;
    // profiling
    bool profile_on = false;
    std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> pending;  // phase, (start, stop)
    std::vector<cudaEvent_t> event_pool;
    sb_profile prof;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    DevBuf<char> flush_buf;
    // scratch reused by reductions / collectives
    DevBuf<char> scratch;
    DevBuf<double> syrk_parts;  // grow-only: per-chunk partial Gram matrices of syrk_tall (dense_own.cu)
    void *pinned = nullptr;  // small pinned staging (4 KB)
    std::vector<double> omega_cache;  // last generated start block (host)
    u64 omega_seed = ~0ull, omega_rows = 0, omega_cols = 0;
    DevBuf<double> omega_dev;         // the same block already in the device layout the n > m branch starts from (m x b, even ld)
    u64 omega_dev_seed = ~0ull, omega_dev_rows = 0, omega_dev_cols = 0;
};

// The packed gene-major entry: x = gene | (cell_local << SB_GENE_BITS), y = count.
#define SB_GENE_BITS 22
#define SB_GENE_MASK 0x3FFFFFu
#define SB_MAX_PANEL_CELLS 1024
#define GA_TBLOCK 16384  // cells per block of the T-side gather order (gather.cu)

// Bit planes of the dense half on the int8 tensor cores (planes.cu)
#define PL_MAX_LEVELS 6
struct PlUnitT {  // T side: a block of 1,024 ranks x up to three levels; CTAs [cta0, cta0 + nctas) stride over the cell tiles
    u32 g0, nlev;
    u32 lev[3], nkb[3];  // level index; 32-gene K blocks of the level inside the block (non-increasing, multiples of 4)
    u32 cta0, nctas;
};
struct PlUnitN {  // N side: a group of 384 ranks; levels 0..nlev-1; CTAs split the cell tiles into contiguous ranges
    u32 g0, nlev;
    u32 mt[PL_MAX_LEVELS];  // 128-gene M tiles of each level inside the group (non-increasing)
    u32 cta0, nctas;
};
struct PlItem {  // T side work item: tiles [t0, t1) of a unit
    u32 unit, t0, t1;
};
struct PlaneSet {
    bool active = false;
    u32 L = 0;
    u32 G[PL_MAX_LEVELS] = {0, 0, 0, 0, 0, 0};  // ranks covered by level k + 1: multiples of 128, non-increasing
    u64 ntiles = 0;                              // cell tiles of 128
    DevBuf<u32> bits[PL_MAX_LEVELS];             // [ntiles][G / 32][128] words
    DevBuf<char> units_t, units_n, items_t, items_n;
    DevBuf<u32> counter;  // work-queue head of the T-side kernel
    // per-pass workspaces, grow-only and kept with the matrix: the digit planes of both sides, the per-unit partial rows of the T side
    // (2.5 GB at C3) and the small scale tables.  Allocating them per pass from the stream-ordered pool works until some other
    // allocation pattern fragments the pool; then these, the largest requests, pay for the remapping.
    mutable DevBuf<signed char> ws_bd, ws_bn;
    mutable DevBuf<double> ws_part, ws_scale2;
    mutable DevBuf<unsigned long long> ws_colmax;
    mutable DevBuf<int> ws_ex;
    u32 n_units_t = 0, n_units_n = 0, n_items_t = 0, n_items_n = 0, t_grid = 0, n_grid = 0;
};

// One side of the panelled gather: the entry stream, its work units and (T side) the gene of every panel slot.
struct GatherLayout {
    bool ready = false;
    u32 rows = 0;     // rows per panel: cells (N side) or gene slots (T side)
    u32 npanels = 0;
    u64 nnz = 0;
    const uint2 *ent = nullptr;  // N side: aliases gm / cold_gm; T side: ent_own
    DevBuf<uint2> ent_own;
    DevBuf<GUnit> units;
    u32 n_units = 0;
    u32 grid = 0;
    DevBuf<u32> cta_first;  // [n_items + 1] first unit of every work item (an item = the units one CTA processes back to back)
    u32 n_items = 0;        // 0: one item per CTA (grid items)
    // Items are handed to the persistent CTAs through a ticket counter: launch i serves tickets [base_i, base_i + n_items) and every
    // CTA draws one failing ticket on its way out, so base advances by n_items + grid per launch and the counter is never reset.
    mutable DevBuf<u32> tickets;
    mutable u32 ticket_base = 0;
    DevBuf<u32> slot_gene;  // T side: [npanels * rows] gene of a slot or 0xFFFFFFFF
};

struct sb_mat {
    sb_ctx *ctx = nullptr;
    u32 m = 0;            // genes
    u64 n = 0;            // local cells
    u64 n_global = 0;     // cells over all ranks
    u64 cell_offset = 0;  // global index of local cell 0
    u64 nnz = 0;          // local non-zeros
    // cell-major copy: cm_ptr[n+1], cm[nnz] = {gene, count}, genes ascending inside a cell
    DevBuf<u64> cm_ptr;
    DevBuf<uint2> cm;
    // gene-major panelled copy: cells are cut into panels of `pc` cells; inside a panel entries are
    // sorted by (gene, cell): gm[k] = {gene | cell_local << 22, count}.  gm_base[np+1] are panel
    // starts.  unit_ptr[np*ur+1] cuts every panel into `ur` gene ranges of similar nnz (work units).
    u32 pc = 0, np = 0, ur = 1;
    DevBuf<uint2> gm;
    DevBuf<u64> gm_base;
    DevBuf<u64> unit_ptr;
    bool have_full_gm = false;  // gm / gm_base above cover ALL entries; built lazily when a dense panel exists
    // Hybrid layout (log-normalization maps only): the `gd` most expressed genes live in a dense u8 panel
    // D[n x gd] (counts 1..SB_DENSE_MAX_COUNT, 0 elsewhere); every other entry -- cold genes and the rare larger
    // counts of hot genes -- stays in the sparse `cold_*` pair of layouts (same formats as cm / gm).
    u32 gd = 0;
    u32 dense_max_count = 15;  // counts 1..dense_max_count live in D
    DevBuf<unsigned char> D;
    DevBuf<u32> hot_idx;      // [gd] gene id of panel column j
    DevBuf<u32> hot_of_gene;  // [m] panel column of a gene or 0xFFFFFFFF
    PlaneSet pl;  // panel_mode 2: bit planes instead of D (gd = ranks of level 1; hot_idx / hot_of_gene are in rank order)
    u64 cold_nnz = 0;
    DevBuf<u64> cold_cm_ptr;
    DevBuf<uint2> cold_cm;
    DevBuf<uint2> cold_gm;
    DevBuf<u64> cold_gm_base;
    // panelled gather layouts over the sparse set the products use (the cold entries when gd > 0, else all entries)
    GatherLayout gn, gt;
    DevBuf<u32> slot_of_gene;  // [m] T-side slot (rank by expression) of a gene
    std::vector<u64> t_seg_len, t_seg_runs;  // T side: entries / runs of every (block, panel) segment, in stream order (host copy for recalibration)
    std::vector<GUnit> t_units_host;         // the T-side units as uploaded
    std::vector<u32> t_first_host;
    std::vector<double> t_rate;              // per-panel rate of the last calibration round (weights the attribution of the next)
    int t_calibrated = 0;                    // calibration rounds done (0: static cost model; >= 1: shares re-cut from a timed pass)
    // cached integer reductions
    DevBuf<u32> cell_tot;
    bool have_cell_tot = false;
};
#define SB_DENSE_MAX_COUNT 15u
#define SB_DENSE_LUT 16

// device view of the per-nonzero map (sqz/src/matrix_map.rs): see MapDev in map.cuh
struct sb_nmat {
    sb_mat *mat = nullptr;
    sb_ctx *ctx = nullptr;  // kept separately: freeing must not touch `mat` (a caller may free the matrix first)
    int kind = 1;      // 1 log chain, 2 binomial deviance, 3 binomial Pearson
    int log_base = 0;  // 0 none, 1 ln, 2 log2, 10 log10
    DevBuf<double> col_scale;  // [n] (kind 1) or binomial n[c]
    DevBuf<double> l1c, inv_l1c;  // [n] kind 1: L_c(1) = log_b(col_scale[c] + 1) and its reciprocal (gather.cu)
    DevBuf<double> lk;            // [n x PL_MAX_LEVELS] kind 1: L_c(k), k = 1 .. 6, finite or 0 (planes.cu: evaluated once per normalize instead of per tile)
    DevBuf<double> row_scale;  // [m] 1/sd (kind 1; may be empty) or binomial pi[r]
    bool has_row_scale = false;
    bool has_offset = false;
    bool v_ones = true;
    DevBuf<double> u;  // [m]
    DevBuf<double> v;  // [n] (only when !v_ones)
};

// ---------------------------------------------------------------- profiling helpers (ctx.cu)
void prof_begin(sb_ctx *ctx, int phase);
void prof_end(sb_ctx *ctx, int phase);
void prof_collect(sb_ctx *ctx);
static inline void count_launch(sb_ctx *ctx, bool own = true) {
    ctx->prof.kernel_launches++;
    if (own) ctx->prof.own_kernel_launches++;
}
struct ProfScope {
    sb_ctx *c;
    int ph;
    ProfScope(sb_ctx *ctx, int phase) : c(ctx), ph(phase) { prof_begin(c, ph); }
    ~ProfScope() { prof_end(c, ph); }
};

int ctx_scratch(sb_ctx *ctx, size_t bytes, void **out);
int comm_allreduce_f64(sb_ctx *ctx, double *buf, size_t count);
int comm_allreduce_u64(sb_ctx *ctx, u64 *buf, size_t count);
int comm_allreduce_max_i32(sb_ctx *ctx, int *host_val);
int comm_allgather_u64_host(sb_ctx *ctx, u64 mine, std::vector<u64> &all);
// every rank takes the same turn before the next collective: a local rejection becomes every rank's error (matrix.cu)
int agree_status(sb_ctx *ctx, int rc, const char *what);
// stable radix sort of (keys, vals) by the 64-bit key; the buffers are replaced by the sorted copies (cluster.cu)
int sort_pairs(sb_ctx *ctx, DevBuf<u64> &keys, DevBuf<u64> &vals, u64 count);
// sSeq pieces shared by diff_exp.cu and merge.cu (diff_exp.cu):
//   one value per local cell -> the values of all cells in global cell order
int gather_cells(sb_ctx *ctx, const std::vector<double> &mine, std::vector<double> &all);
//   params for this matrix and context (sizes, NULL arrays)
int sseq_check_params(sb_mat *mat, const sb_sseq_params *p, const char *fn);
//   per-group gene sums of the whole matrix into acc[n_groups x m] (replicated over ranks); d_lab: this rank's labels on the device
int group_gene_sums(sb_mat *mat, const u32 *d_lab, u32 n_groups, DevBuf<u64> &acc);
//   the pairwise test stage: comparison j is row rows[2j] of d_sums[. x m] against row rows[2j + 1], with s_in[j] / s_out[j]
int sseq_pair_tests(sb_mat *mat, const sb_sseq_params *prm, const u64 *d_sums, const std::vector<u32> &rows, const std::vector<double> &s_in,
                    const std::vector<double> &s_out, u64 big_count, sb_diff_exp_out *out);
// rows [n_local x width] of every rank, in global cell order, into dst (32-bit words; counts from comm_allgather_u64_host) (umap.cu)
int um_gather_rows(sb_ctx *ctx, const void *mine_h, u64 n_local, u64 width_words, const std::vector<u64> &counts, u64 maxr, u32 *dst);
// kNN-graph pieces shared by umap.cu and tsne.cu (defined in umap.cu):
//   SplitMix64's finaliser, the counter hash of negative samples and random starts
__host__ __device__ __forceinline__ u64 um_mix64(u64 z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
//   thread per (row, slot) of nbr [n x k] (0xFFFFFFFF pads a row's end): err bits 1 index >= n, 2 self index, 4 duplicate in the
//   row, 8 padding before the row end; d = sqrt(sum_c (x_j,c - x_i,c)^2) in coordinate order without contraction (0 at padding)
__global__ void k_um_dist(const double *__restrict__ X, const u32 *__restrict__ nbr, u64 n, u32 dim, u32 k, double *__restrict__ d,
                          int *__restrict__ err);
//   a weighted graph on the device: symmetric CSR, columns ascending, f64 weights in (0, 1]
struct UmGraph {
    u64 n = 0, nnz = 0;
    DevBuf<u64> ptr;     // [n + 1]
    DevBuf<u32> idx;     // [nnz]
    DevBuf<double> w;    // [nnz]
};
//   the flagged entries of in[count] into out, their number into *d_num (device); T = u32, u64 or double
template <typename T>
int um_select(sb_ctx *ctx, const T *in, const char *flags, T *out, u64 count, u64 *d_num);
//   keys (row << 32 | col, ascending) of g.nnz entries -> g.ptr, g.idx
int um_rows_from_keys(sb_ctx *ctx, const u64 *keys, UmGraph &g);
//   a host CSR of n vertices: n < 2^32 - 1, indptr from 0 and non-decreasing, arrays present when there are entries
int um_csr_host_check(u64 n, const u64 *indptr, const u32 *indices, const double *weights, const char *fn);
//   the host CSR (checked above) to g, validated on the device: column < n, weights in (0, 1], no duplicate, symmetric with equal
//   weights both ways (SB_ERR_INVALID_ARG otherwise); columns ascending in g; trace: the name of the validation's trace scope
int um_csr_upload(sb_ctx *ctx, u64 n, const u64 *indptr, const u32 *indices, const double *weights, UmGraph &g, const char *fn,
                  const char *trace);
// percentile_of_sorted (stat.rs:140-163) at the fraction q: rank q (n - 1), linear interpolation; sorts v (moments.cu)
double percentile_of(std::vector<double> &v, double q);

// every API entry: select the device and publish the stream used for stream-ordered allocations
#define SB_ENTER(ctx_ptr)                         \
    do {                                          \
        SB_CUDA(cudaSetDevice((ctx_ptr)->device)); \
        sb_set_alloc_stream((ctx_ptr)->stream, (ctx_ptr)->pool); \
    } while (0)

// SCANB200_TRACE=1: host wall-clock trace of the upload / build stages (synchronising; diagnostics only)
struct TraceScope {
    sb_ctx *c;
    const char *name;
    double t0;
    static bool on();
    static int level();
    static double now();
    TraceScope(sb_ctx *ctx, const char *n) : c(ctx), name(n), t0(0) {
        if (on()) {
            cudaStreamSynchronize(c->stream);
            t0 = now();
        }
    }
    ~TraceScope() {
        if (on()) {
            cudaStreamSynchronize(c->stream);
            fprintf(stderr, "[scanb200] %-28s %8.2f ms\n", name, (now() - t0) * 1e3);
        }
    }
};

// Build-time stages (upload, layout construction): always drain the library stream at both ends, trace or not.  Measured
// on the 1.3M-cell upload: with these synchronisations every call takes 93.5 ms; without them the host runs ahead of the
// device, the stream-ordered pool grows (reserved memory climbs call after call) and calls take 95-780 ms.
struct SyncScope {
    sb_ctx *c;
    const char *name;
    double t0;
    SyncScope(sb_ctx *ctx, const char *n) : c(ctx), name(n), t0(0) {
        cudaStreamSynchronize(c->stream);
        if (TraceScope::on()) t0 = TraceScope::now();
    }
    ~SyncScope() {
        cudaStreamSynchronize(c->stream);
        if (TraceScope::on()) fprintf(stderr, "[scanb200] %-28s %8.2f ms\n", name, (TraceScope::now() - t0) * 1e3);
    }
};

static inline unsigned cdiv(u64 a, u64 b) { return (unsigned)((a + b - 1) / b); }
