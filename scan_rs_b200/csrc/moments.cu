// moments.cu -- the per-gene / per-cell moment consumers of the count matrix that diff-exp reads (SURVEY 8f rank 4):
//   mean_var_axis   sqz/src/mat.rs:285-329          mean_var_rows   mat.rs:332-374
//   sum_cols        mat.rs:414-446                  sum_rows        mat.rs:449-476          sum_rows_dual  mat.rs:484-583
//   size_factors    diff-exp/src/diff_exp.rs:314-334 (median = 50th percentile with linear interpolation, diff-exp/src/stat.rs:107-163)
// applied to raw counts or to the SizeNormalized view `v as f64 / size_factor[c]` (diff_exp.rs:340-358; NaN factors become 0).
// One kernel serves all of them: a warp per cell over the cell-major stream, per-gene accumulators updated with reductions.
// Raw counts accumulate in u64 (exact: identical to the reference's f64 sums of integers below 2^53); the SizeNormalized
// view accumulates in f64 with reductions whose order varies from run to run (bar: 1e-12 relative, tests/test_gpu_parity.py).
// Sharded contexts: cell index lists are LOCAL to the rank's shard; per-gene results are summed over ranks.
#include <cmath>

#include "common.cuh"

int mat_cell_totals_dev(sb_mat *mat);

static inline int mo_grid(sb_ctx *ctx, u64 cells) { return (int)std::max<u64>(1, std::min<u64>((cells * 32 + 255) / 256, (u64)ctx->sm_count * 16)); }

// w1 / w2: multiplicity of a cell in the first / second index list (NULL: every cell once / list absent)
__global__ void k_mo_int(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, const u32 *__restrict__ w1, const u32 *__restrict__ w2,
                         int square2, unsigned long long *__restrict__ out1, unsigned long long *__restrict__ out2) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        const u32 m1 = w1 ? w1[c] : 1u, m2 = square2 ? m1 : (w2 ? w2[c] : 0u);
        if (!m1 && !m2) continue;
        const u64 s = ptr[c], e = ptr[c + 1];
        for (u64 k = s + lane; k < e; k += 32) {
            const uint2 z = cm[k];
            if (m1) atomicAdd(&out1[z.x], (unsigned long long)z.y * m1);
            if (m2 && out2) atomicAdd(&out2[z.x], (square2 ? (unsigned long long)z.y * z.y : (unsigned long long)z.y) * m2);
        }
    }
}

// SizeNormalized view: x = v / div[c]; axis 1 (per gene): S1[g] += w x, S2[g] += w x^2; axis 0 (per cell): plain per-cell sums
__global__ void k_mo_f64_genes(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, const double *__restrict__ div, const u32 *__restrict__ w1,
                               double *__restrict__ S1, double *__restrict__ S2) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        const u32 m1 = w1 ? w1[c] : 1u;
        if (!m1) continue;
        const double d = div[c], wd = (double)m1;
        const u64 s = ptr[c], e = ptr[c + 1];
        for (u64 k = s + lane; k < e; k += 32) {
            const uint2 z = cm[k];
            const double x = (double)z.y / d;  // a division, as SizeNormalized::map (diff_exp.rs:350-352)
            atomicAdd(&S1[z.x], wd * x);
            atomicAdd(&S2[z.x], wd * (x * x));
        }
    }
}
__global__ void k_mo_f64_cells(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, const double *__restrict__ div, double *__restrict__ S1,
                               double *__restrict__ S2) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        const double d = div ? div[c] : 1.0;
        const u64 s = ptr[c], e = ptr[c + 1];
        double a = 0.0, b = 0.0;
        for (u64 k = s + lane; k < e; k += 32) {
            const double x = (double)cm[k].y / d;
            a += x;
            b += x * x;
        }
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, o);
            b += __shfl_xor_sync(0xffffffffu, b, o);
        }
        if (lane == 0) {
            S1[c] = a;
            S2[c] = b;
        }
    }
}

// multiplicities of the local cells in an index list (mat.rs:362-369: the CSC branch walks a listed column once per listing)
static int upload_weights(sb_mat *mat, const uint64_t *cols, uint64_t n_cols, DevBuf<u32> &w) {
    sb_ctx *ctx = mat->ctx;
    std::vector<u32> h(std::max<u64>(mat->n, 1), 0u);
    for (u64 i = 0; i < n_cols; i++) {
        if (cols[i] >= mat->n) return sb_fail(SB_ERR_INVALID_ARG, "cell index %llu out of range (%llu local cells)", (unsigned long long)cols[i], (unsigned long long)mat->n);
        h[cols[i]]++;
    }
    SB_TRY(w.alloc(h.size()));
    SB_CUDA(cudaMemcpyAsync(w.p, h.data(), h.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// SizeNormalized::new (diff_exp.rs:341-344): NaN -> 0
static int upload_div(sb_mat *mat, const double *cell_div, DevBuf<double> &d) {
    sb_ctx *ctx = mat->ctx;
    std::vector<double> h(std::max<u64>(mat->n, 1), 1.0);
    for (u64 i = 0; i < mat->n; i++) h[i] = cell_div[i] != cell_div[i] ? 0.0 : cell_div[i];
    SB_TRY(d.alloc(h.size()));
    SB_CUDA(cudaMemcpyAsync(d.p, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// per-gene first / second moments over the selected cells -> mean, var (V[X] = E[X^2] - E[X]^2, mat.rs:322-327)
static int gene_mean_var(sb_mat *mat, const DevBuf<u32> *w, const double *cell_div, double count, double *mean, double *var) {
    sb_ctx *ctx = mat->ctx;
    const u32 m = mat->m;
    std::vector<double> s1(m), s2(m);
    if (!cell_div) {
        DevBuf<u64> acc;
        SB_TRY(acc.alloc((size_t)2 * m));
        SB_CUDA(cudaMemsetAsync(acc.p, 0, (size_t)2 * m * sizeof(u64), ctx->stream));
        if (mat->n && mat->nnz) {
            ProfScope ps(ctx, PH_REDUCE);
            k_mo_int<<<mo_grid(ctx, mat->n), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, w ? w->p : nullptr, nullptr, 1,
                                                                    (unsigned long long *)acc.p, (unsigned long long *)acc.p + m);
            count_launch(ctx);
        }
        SB_TRY(comm_allreduce_u64(ctx, acc.p, (size_t)2 * m));
        std::vector<u64> h((size_t)2 * m);
        SB_CUDA(cudaMemcpyAsync(h.data(), acc.p, h.size() * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        for (u32 g = 0; g < m; g++) {
            s1[g] = (double)h[g];
            s2[g] = (double)h[m + g];
        }
    } else {
        DevBuf<double> acc, d;
        SB_TRY(upload_div(mat, cell_div, d));
        SB_TRY(acc.alloc((size_t)2 * m));
        SB_CUDA(cudaMemsetAsync(acc.p, 0, (size_t)2 * m * sizeof(double), ctx->stream));
        if (mat->n && mat->nnz) {
            ProfScope ps(ctx, PH_MOMENTS);
            k_mo_f64_genes<<<mo_grid(ctx, mat->n), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, d.p, w ? w->p : nullptr, acc.p, acc.p + m);
            count_launch(ctx);
        }
        SB_TRY(comm_allreduce_f64(ctx, acc.p, (size_t)2 * m));
        SB_CUDA(cudaMemcpyAsync(s1.data(), acc.p, m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(s2.data(), acc.p + m, m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    for (u32 g = 0; g < m; g++) {
        const double mu = s1[g] / count;
        mean[g] = mu;
        var[g] = s2[g] / count - mu * mu;
    }
    return SB_OK;
}

// sums the listed (local) counts over ranks
static int global_count(sb_ctx *ctx, u64 local, double *out) {
    if (ctx->nranks == 1) {
        *out = (double)local;
        return SB_OK;
    }
    std::vector<u64> all;
    SB_TRY(comm_allgather_u64_host(ctx, local, all));
    u64 t = 0;
    for (u64 x : all) t += x;
    *out = (double)t;
    return SB_OK;
}

extern "C" int sb_mean_var_axis(sb_mat *mat, int axis, const double *cell_div, double *mean, double *var) {
    if (!mat || !mean || !var || (axis != 0 && axis != 1)) return sb_fail(SB_ERR_INVALID_ARG, "sb_mean_var_axis: bad argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    if (axis == 1) return gene_mean_var(mat, nullptr, cell_div, (double)mat->n_global, mean, var);  // per gene, over all cells
    // per cell, over the m genes: shard-local
    DevBuf<double> acc, d;
    if (cell_div) SB_TRY(upload_div(mat, cell_div, d));
    SB_TRY(acc.alloc(std::max<u64>(1, 2 * mat->n)));
    if (mat->n) {
        ProfScope ps(ctx, PH_MOMENTS);
        k_mo_f64_cells<<<mo_grid(ctx, mat->n), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, cell_div ? d.p : nullptr, acc.p, acc.p + mat->n);
        count_launch(ctx);
        SB_CUDA(cudaMemcpyAsync(mean, acc.p, mat->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(var, acc.p + mat->n, mat->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    const double mm = (double)mat->m;
    for (u64 c = 0; c < mat->n; c++) {
        const double mu = mean[c] / mm;
        mean[c] = mu;
        var[c] = var[c] / mm - mu * mu;
    }
    return SB_OK;
}

extern "C" int sb_mean_var_rows(sb_mat *mat, const uint64_t *cols, uint64_t n_cols, const double *cell_div, double *mean, double *var) {
    if (!mat || !mean || !var || (!cols && n_cols)) return sb_fail(SB_ERR_INVALID_ARG, "sb_mean_var_rows: bad argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    DevBuf<u32> w;
    SB_TRY(upload_weights(mat, cols, n_cols, w));
    double count = 0.0;
    SB_TRY(global_count(ctx, n_cols, &count));
    return gene_mean_var(mat, &w, cell_div, count, mean, var);
}

static int sum_rows_impl(sb_mat *mat, const uint64_t *cols1, uint64_t n1, const uint64_t *cols2, uint64_t n2, bool dual, uint64_t *sum1, uint64_t *sum2) {
    sb_ctx *ctx = mat->ctx;
    const u32 m = mat->m;
    DevBuf<u32> w1, w2;
    SB_TRY(upload_weights(mat, cols1, n1, w1));
    if (dual) SB_TRY(upload_weights(mat, cols2, n2, w2));
    DevBuf<u64> acc;
    SB_TRY(acc.alloc((size_t)2 * m));
    SB_CUDA(cudaMemsetAsync(acc.p, 0, (size_t)2 * m * sizeof(u64), ctx->stream));
    if (mat->n && mat->nnz) {
        ProfScope ps(ctx, PH_REDUCE);
        k_mo_int<<<mo_grid(ctx, mat->n), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, w1.p, dual ? w2.p : nullptr, 0, (unsigned long long *)acc.p,
                                                                (unsigned long long *)acc.p + m);
        count_launch(ctx);
    }
    SB_TRY(comm_allreduce_u64(ctx, acc.p, (size_t)2 * m));
    SB_CUDA(cudaMemcpyAsync(sum1, acc.p, m * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    if (dual) SB_CUDA(cudaMemcpyAsync(sum2, acc.p + m, m * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

extern "C" int sb_sum_rows(sb_mat *mat, const uint64_t *cols, uint64_t n_cols, uint64_t *out_m) {
    if (!mat || !out_m || (!cols && n_cols)) return sb_fail(SB_ERR_INVALID_ARG, "sb_sum_rows: bad argument");
    SB_ENTER(mat->ctx);
    return sum_rows_impl(mat, cols, n_cols, nullptr, 0, false, out_m, nullptr);
}

// merge_join_by over two sorted lists (mat.rs:516-553): a cell in both lists adds to both sums
extern "C" int sb_sum_rows_dual(sb_mat *mat, const uint64_t *cols1, uint64_t n1, const uint64_t *cols2, uint64_t n2, uint64_t *sum1, uint64_t *sum2) {
    if (!mat || !sum1 || !sum2 || (!cols1 && n1) || (!cols2 && n2)) return sb_fail(SB_ERR_INVALID_ARG, "sb_sum_rows_dual: bad argument");
    SB_ENTER(mat->ctx);
    return sum_rows_impl(mat, cols1, n1, cols2, n2, true, sum1, sum2);
}

// sum_cols (mat.rs:414-446): the totals of the listed cells, in list order
extern "C" int sb_sum_cols(sb_mat *mat, const uint64_t *cols, uint64_t n_cols, uint64_t *out) {
    if (!mat || (!out && n_cols) || (!cols && n_cols)) return sb_fail(SB_ERR_INVALID_ARG, "sb_sum_cols: bad argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    DevBuf<double> acc;
    SB_TRY(acc.alloc(std::max<u64>(1, 2 * mat->n)));
    std::vector<double> h(mat->n);
    if (mat->n) {
        k_mo_f64_cells<<<mo_grid(ctx, mat->n), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, nullptr, acc.p, acc.p + mat->n);
        count_launch(ctx);
        SB_CUDA(cudaMemcpyAsync(h.data(), acc.p, mat->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    for (u64 i = 0; i < n_cols; i++) {
        if (cols[i] >= mat->n) return sb_fail(SB_ERR_INVALID_ARG, "sb_sum_cols: cell index out of range");
        out[i] = (uint64_t)h[cols[i]];  // sums of integers below 2^53: exact
    }
    return SB_OK;
}

// percentile_of_sorted (stat.rs:140-163) at the fraction q in [0, 1]: rank q (n - 1), linear interpolation; sorts v (non-empty).
// The median of the size factors is q = 0.5; sSeq's zeta_hat (diff_exp.cu) is q = zeta_quantile.
double percentile_of(std::vector<double> &v, double q) {
    std::sort(v.begin(), v.end());
    if (v.size() == 1) return v[0];
    const double rank = q * (double)(v.size() - 1);
    const double lr = std::floor(rank), d = rank - lr;
    const size_t i = (size_t)lr;
    if (i + 1 >= v.size()) return v[i];
    return v[i] + (v[i + 1] - v[i]) * d;
}
static double percentile_median(std::vector<double> &v) { return percentile_of(v, 0.5); }

// size_factors (diff_exp.rs:314-334).  cells (local indices, may be NULL = all cells) select the cells whose totals define the
// median; umi_counts (may be NULL) replaces the totals: one value per listed cell (or per local cell when cells is NULL).
// out[n_local]: counts / median at the listed cells, 0 elsewhere (every cell when cells is NULL).
extern "C" int sb_size_factors(sb_mat *mat, const uint64_t *cells, uint64_t n_cells, const double *umi_counts, double *out) {
    if (!mat || (!out && mat->n) || (!cells && n_cells)) return sb_fail(SB_ERR_INVALID_ARG, "sb_size_factors: bad argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    const u64 cnt = cells ? n_cells : mat->n;
    std::vector<double> cpc(cnt);
    if (umi_counts) {
        for (u64 i = 0; i < cnt; i++) cpc[i] = umi_counts[i];
    } else {
        DevBuf<double> acc;
        SB_TRY(acc.alloc(std::max<u64>(1, 2 * mat->n)));
        std::vector<double> h(mat->n);
        if (mat->n) {
            k_mo_f64_cells<<<mo_grid(ctx, mat->n), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, nullptr, acc.p, acc.p + mat->n);
            count_launch(ctx);
            SB_CUDA(cudaMemcpyAsync(h.data(), acc.p, mat->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        }
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        for (u64 i = 0; i < cnt; i++) {
            const u64 c = cells ? cells[i] : i;
            if (c >= mat->n) return sb_fail(SB_ERR_INVALID_ARG, "sb_size_factors: cell index out of range");
            cpc[i] = h[c];
        }
    }
    // the median is over the listed cells of ALL ranks: gather the counts (zero-padded all-reduce of one slot per rank's cell)
    std::vector<double> all;
    if (ctx->nranks > 1) {
        std::vector<u64> counts;
        SB_TRY(comm_allgather_u64_host(ctx, cnt, counts));
        u64 total = 0, off = 0;
        for (int r = 0; r < ctx->nranks; r++) {
            if (r < ctx->rank) off += counts[r];
            total += counts[r];
        }
        all.assign(total, 0.0);
        std::copy(cpc.begin(), cpc.end(), all.begin() + off);
        DevBuf<double> d;
        SB_TRY(d.alloc(std::max<u64>(1, total)));
        if (total) SB_CUDA(cudaMemcpyAsync(d.p, all.data(), total * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        SB_TRY(comm_allreduce_f64(ctx, d.p, total));
        if (total) SB_CUDA(cudaMemcpyAsync(all.data(), d.p, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    } else {
        all = cpc;
    }
    if (all.empty()) return sb_fail(SB_ERR_INVALID_ARG, "sb_size_factors: no cells (the reference asserts a non-empty sample, stat.rs:144)");
    const double med = percentile_median(all);
    for (u64 c = 0; c < mat->n; c++) out[c] = 0.0;
    for (u64 i = 0; i < cnt; i++) out[cells ? cells[i] : i] = cpc[i] / med;
    return SB_OK;
}
