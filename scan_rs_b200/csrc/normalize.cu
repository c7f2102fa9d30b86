// normalize.cu -- builds the device-side LowRankOffset: column scales from the integer cell
// totals, per-gene moments of the log-normalized values (K5), 1/sd row scales and the -mean/sd
// offset vector.  Restates scan-rs/src/normalization.rs:46-213 (+ :218-323 for the binomial
// residual kinds) and sqz/src/mat.rs:937-1001.
#include "common.cuh"
#include "map.cuh"

int mat_cell_totals_dev(sb_mat *mat);
int mat_median_total(sb_mat *mat, u32 *median, int *nonempty);
int mat_gene_sums_dev(sb_mat *mat, int mode, const unsigned char *excl_cells, const unsigned char *excl_genes, u64 *d_out, bool allreduce);
int spmm_t(sb_nmat *a, const double *Y, u32 ldy, u32 w, double *out, u32 ldo, double *uy_scratch);
int spmm_n(sb_nmat *a, const double *X, u32 ldx, u32 w, double *P, u32 ldp);
int dense_moments(sb_nmat *a, double *S1, double *S2);
int mat_ensure_full_gm(sb_mat *mt);

#define FULLMASK 0xffffffffu

// col_scales[c] = target / (count[c] as f64)   (normalization.rs:169)
__global__ void k_col_scale(const u32 *__restrict__ counts, u64 n, double target, double *__restrict__ out) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = target / (double)counts[i];
}

// L_c(1) = log_b(cs_c * 1 + 1), the map value of a count of 1, and its reciprocal: the panelled gather stages operand
// rows pre-multiplied by it (N side) or applies it once per run (T side) instead of once per entry.  Same function of
// the same inputs as the per-entry evaluation, so the bits agree.
__global__ void k_l1_tables(const double *__restrict__ cs, u64 n, int log_base, double *__restrict__ l1, double *__restrict__ inv) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const double v = map_log_part(log_base, cs[i], 1u, sb_log_table);
        l1[i] = v;
        const double r = 1.0 / v;
        inv[i] = (v != 0.0 && r == r && r - r == 0.0) ? r : 0.0;
    }
}

// lk[c * PL_MAX_LEVELS + k - 1] = L_c(k) for the count levels the bit planes can hold; non-finite values (a zero total gives an
// infinite, never-used column scale, normalization.rs:169) are stored as 0, as the plane kernels want them
__global__ void k_level_table(const double *__restrict__ cs, u64 n, int log_base, double *__restrict__ lk) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * PL_MAX_LEVELS) return;
    const u64 c = i / PL_MAX_LEVELS;
    const u32 k = (u32)(i - c * PL_MAX_LEVELS) + 1u;
    const double v = map_log_part(log_base, cs[c], k, sb_log_table);
    lk[i] = (v == v && fabs(v) < 1.0e300) ? v : 0.0;
}

__global__ void k_fill(double *p, u64 n, double v) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// K5: S1[g] = sum_c L_gc, S2[g] = sum_c L_gc^2 with L = log_b(cs_c * v + 1) over the gene-major
// panelled stream.  A warp reads 32 consecutive entries (sorted by gene), does a segmented
// warp reduction keyed on the gene and the segment tails add into S with f64 reductions.
__global__ void __launch_bounds__(256) k_moments(const uint2 *__restrict__ gm, const u64 *__restrict__ gm_base, u32 np, u32 pc,
                                                  int log_base, const double *__restrict__ col, double *__restrict__ S1,
                                                  double *__restrict__ S2) {
    const int lane = threadIdx.x & 31;
    const u32 wpb = blockDim.x >> 5;
    for (u32 p = blockIdx.y; p < np; p += gridDim.y) {
        const u64 pb = gm_base[p], pe = gm_base[p + 1];
        const u64 cell0 = (u64)p * pc;
        for (u64 k0 = pb + ((u64)blockIdx.x * wpb + (threadIdx.x >> 5)) * 32; k0 < pe; k0 += (u64)gridDim.x * wpb * 32) {
            const u64 k = k0 + lane;
            const bool valid = k < pe;
            uint2 z = valid ? gm[k] : make_uint2(0xFFFFFFFFu, 0u);
            const u32 gene = z.x & SB_GENE_MASK, cl = z.x >> SB_GENE_BITS;
            double l1 = 0.0, l2 = 0.0;
            if (valid) {
                l1 = map_log_part(log_base, col[cell0 + cl], z.y, sb_log_table);
                l2 = l1 * l1;
            }
            const u32 key = valid ? gene : 0xFFFFFFFFu;
            // segmented inclusive scan over equal keys (keys are sorted inside the chunk)
            for (int o = 1; o < 32; o <<= 1) {
                double t1 = __shfl_up_sync(FULLMASK, l1, o);
                double t2 = __shfl_up_sync(FULLMASK, l2, o);
                u32 ko = __shfl_up_sync(FULLMASK, key, o);
                if (lane >= o && ko == key) {
                    l1 += t1;
                    l2 += t2;
                }
            }
            u32 knext = __shfl_down_sync(FULLMASK, key, 1);
            if (valid && (lane == 31 || knext != key)) {
                atomicAdd(S1 + gene, l1);
                atomicAdd(S2 + gene, l2);
            }
        }
    }
}

// scale_and_center (mat.rs:986-1001) on the reduced moments:
//   mean = S1/n; sd = sqrt(S2/n - mean^2) or 1.0 if that is <= 0 (:996); mean /= sd (:998);
//   row_scale = 1/sd (:970); u = -(mean/sd) (:946)
__global__ void k_finish_moments(const double *__restrict__ S1, const double *__restrict__ S2, u32 m, double n_cells,
                                 const double *__restrict__ sd_override, double *__restrict__ row_scale, double *__restrict__ u) {
    u32 g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < m) {
        double mean = S1[g] / n_cells;
        double sd;
        if (sd_override) {
            sd = sd_override[g];
        } else {
            double sq = S2[g] / n_cells;
            double x = sq - mean * mean;
            sd = x <= 0.0 ? 1.0 : sqrt(x);
        }
        mean = mean / sd;
        row_scale[g] = 1.0 / sd;
        u[g] = -mean;
    }
}

// S[0, m) = S1, S[m, 2m) = S2, all-reduced over ranks (also reached by tests/cuda/spmm_harness.cu)
int nmat_moments(sb_nmat *a, double *S /* 2m */) {
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    SB_CUDA(cudaMemsetAsync(S, 0, 2 * (size_t)mt->m * sizeof(double), ctx->stream));
    const bool hybrid = mt->gd > 0;  // moments are only taken of log-normalized (kind 1) matrices
    if (!hybrid) SB_TRY(mat_ensure_full_gm(mt));
    const uint2 *gm = hybrid ? mt->cold_gm.p : mt->gm.p;
    const u64 *gm_base = hybrid ? mt->cold_gm_base.p : mt->gm_base.p;
    if (mt->nnz) {
        ProfScope ps(ctx, PH_MOMENTS);
        u32 gy = mt->np < 65535u ? mt->np : 65535u;
        u32 gx = (u32)((u64)ctx->sm_count * 16 / gy);
        if (gx < 1) gx = 1;
        dim3 grid(gx, gy);
        if (hybrid ? mt->cold_nnz : mt->nnz) {
            k_moments<<<grid, 256, 0, ctx->stream>>>(gm, gm_base, mt->np, mt->pc, a->log_base, a->col_scale.p, S, S + mt->m);
            count_launch(ctx);
        }
        if (hybrid) SB_TRY(dense_moments(a, S, S + mt->m));
        SB_CUDA(cudaGetLastError());
    }
    SB_TRY(comm_allreduce_f64(ctx, S, 2 * (size_t)mt->m));
    return SB_OK;
}

// sum_g ( rs_g^2 S2_g + 2 u_g rs_g S1_g + n u_g^2 ): the squared Frobenius norm of S + u 1^T from the gene moments
__global__ void k_frob_from_moments(const double *__restrict__ S1, const double *__restrict__ S2, const double *__restrict__ rs,
                                    const double *__restrict__ u, u32 m, double n, double *__restrict__ out) {
    double acc = 0.0;
    for (u32 g = blockIdx.x * blockDim.x + threadIdx.x; g < m; g += gridDim.x * blockDim.x) {
        const double r = rs ? rs[g] : 1.0, ug = u ? u[g] : 0.0;
        acc += r * r * S2[g] + 2.0 * ug * r * S1[g] + n * ug * ug;
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

extern "C" int sb_nmat_frobenius_sq(sb_nmat *a, double *out) {
    if (!a || !out) return sb_fail(SB_ERR_INVALID_ARG, "sb_nmat_frobenius_sq: NULL argument");
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    SB_ENTER(ctx);
    if (a->kind != 1 || !a->v_ones) return sb_fail(SB_ERR_UNSUPPORTED, "sb_nmat_frobenius_sq: log-chain normalizations only");
    DevBuf<double> S, acc;
    SB_TRY(S.alloc(2 * (size_t)mt->m + 1));
    SB_TRY(acc.alloc(1));
    SB_TRY(nmat_moments(a, S.p));  // all-reduced over ranks
    SB_CUDA(cudaMemsetAsync(acc.p, 0, sizeof(double), ctx->stream));
    if (mt->m) {
        k_frob_from_moments<<<cdiv(mt->m, 256), 256, 0, ctx->stream>>>(S.p, S.p + mt->m, a->has_row_scale ? a->row_scale.p : nullptr,
                                                                       a->has_offset ? a->u.p : nullptr, mt->m, (double)mt->n_global, acc.p);
        count_launch(ctx);
    }
    SB_CUDA(cudaMemcpyAsync(out, acc.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// col_scale = target / (size factor or cell total) per local cell (normalization.rs:169), and the L_c(1) and level tables of it
static int log_col_tables(sb_nmat *a, double target, const uint32_t *size_factors) {
    sb_mat *mat = a->mat;
    sb_ctx *ctx = mat->ctx;
    a->target = target;
    a->like_ok = size_factors == nullptr;
    SB_TRY(a->col_scale.alloc(mat->n));
    if (mat->n) {
        const u32 *counts = mat->cell_tot.p;
        DevBuf<u32> d_sf;
        if (size_factors) {
            SB_TRY(d_sf.alloc(mat->n));
            SB_CUDA(cudaMemcpyAsync(d_sf.p, size_factors, mat->n * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
            counts = d_sf.p;
        }
        k_col_scale<<<cdiv(mat->n, 256), 256, 0, ctx->stream>>>(counts, mat->n, target, a->col_scale.p);
        SB_TRY(a->l1c.alloc(mat->n));
        SB_TRY(a->inv_l1c.alloc(mat->n));
        k_l1_tables<<<cdiv(mat->n, 256), 256, 0, ctx->stream>>>(a->col_scale.p, mat->n, a->log_base, a->l1c.p, a->inv_l1c.p);
        SB_TRY(a->lk.alloc(mat->n * PL_MAX_LEVELS));
        k_level_table<<<cdiv(mat->n * PL_MAX_LEVELS, 256), 256, 0, ctx->stream>>>(a->col_scale.p, mat->n, a->log_base, a->lk.p);
        count_launch(ctx);
        count_launch(ctx); count_launch(ctx);
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return SB_OK;
}

extern "C" int sb_log_normalize(sb_mat *mat, int has_target, double target, int log_base, const uint32_t *size_factors,
                                int center_scale, const double *sd_override, sb_nmat **out) {
    if (!mat || !out) return sb_fail(SB_ERR_INVALID_ARG, "sb_log_normalize: NULL argument");
    if (log_base != 0 && log_base != SB_LOG_E && log_base != SB_LOG_TWO && log_base != SB_LOG_TEN)
        return sb_fail(SB_ERR_INVALID_ARG, "sb_log_normalize: bad log base %d", log_base);
    if (center_scale < 0 || center_scale > 2 || (center_scale == 2 && !sd_override))
        return sb_fail(SB_ERR_INVALID_ARG, "sb_log_normalize: bad center_scale");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    *out = nullptr;
    std::unique_ptr<sb_nmat> a(new sb_nmat());
    a->mat = mat;
    a->ctx = mat->ctx;
    a->kind = 1;
    a->log_base = log_base;
    // normalization.rs:148-168
    SB_TRY(mat_cell_totals_dev(mat));
    if (!has_target) {
        u32 med = 0;
        int nonempty = 0;
        SB_TRY(mat_median_total(mat, &med, &nonempty));
        target = nonempty ? ((double)med > 1.0 ? (double)med : 1.0) : 1.0;  // .max(1.0), map_or(1.0)
    }
    SB_TRY(log_col_tables(a.get(), target, size_factors));
    if (center_scale) {
        DevBuf<double> S, sd;
        SB_TRY(S.alloc(2 * (size_t)mat->m));
        SB_TRY(nmat_moments(a.get(), S.p));
        if (center_scale == 2) {
            SB_TRY(sd.alloc(mat->m));
            SB_CUDA(cudaMemcpyAsync(sd.p, sd_override, (size_t)mat->m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        }
        SB_TRY(a->row_scale.alloc(mat->m));
        SB_TRY(a->u.alloc(mat->m));
        if (mat->m) {
            k_finish_moments<<<cdiv(mat->m, 256), 256, 0, ctx->stream>>>(S.p, S.p + mat->m, mat->m, (double)mat->n_global,
                                                                          center_scale == 2 ? sd.p : nullptr, a->row_scale.p, a->u.p);
            count_launch(ctx);
        }
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        a->has_row_scale = true;
        a->has_offset = true;
        a->v_ones = true;
    }
    *out = a.release();
    return SB_OK;
}

// binomial residual constructors (normalization.rs:218-260, 307-323)
__global__ void k_binom_params(const unsigned long long *__restrict__ gene_tot, u32 m, double total, int deviance,
                               double *__restrict__ pi, double *__restrict__ u) {
    u32 g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g < m) {
        double x = (double)gene_tot[g] / total;
        pi[g] = x;
        u[g] = deviance ? sqrt(log(1.0 / (1.0 - x))) : sqrt(x / (1.0 - x));
    }
}

__global__ void k_binom_cells(const u32 *__restrict__ cell_tot, u64 n, int deviance, double *__restrict__ nn, double *__restrict__ v) {
    u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n) {
        double x = (double)cell_tot[c];
        nn[c] = x;
        v[c] = deviance ? -sqrt(2.0 * x) : -sqrt(x);
    }
}

static int normalize_binomial(sb_mat *mat, int deviance, sb_nmat **out) {
    sb_ctx *ctx = mat->ctx;
    std::unique_ptr<sb_nmat> a(new sb_nmat());
    a->mat = mat;
    a->ctx = mat->ctx;
    a->kind = deviance ? 2 : 3;
    a->log_base = 0;
    SB_TRY(mat_cell_totals_dev(mat));
    DevBuf<u64> gt;
    SB_TRY(gt.alloc(mat->m));
    SB_TRY(mat_gene_sums_dev(mat, 0, nullptr, nullptr, gt.p, true));
    std::vector<u64> h(mat->m);
    if (mat->m) SB_CUDA(cudaMemcpyAsync(h.data(), gt.p, (size_t)mat->m * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    // total_umi_count = n.sum(): integer-valued f64 sums are exact below 2^53 (normalization.rs:224-225)
    u64 total = 0;
    for (u64 x : h) total += x;
    SB_TRY(a->col_scale.alloc(mat->n));
    SB_TRY(a->row_scale.alloc(mat->m));
    SB_TRY(a->u.alloc(mat->m));
    SB_TRY(a->v.alloc(mat->n));
    if (mat->m) {
        k_binom_params<<<cdiv(mat->m, 256), 256, 0, ctx->stream>>>((unsigned long long *)gt.p, mat->m, (double)total, deviance, a->row_scale.p, a->u.p);
        count_launch(ctx);
    }
    if (mat->n) {
        k_binom_cells<<<cdiv(mat->n, 256), 256, 0, ctx->stream>>>(mat->cell_tot.p, mat->n, deviance, a->col_scale.p, a->v.p);
        count_launch(ctx);
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    a->has_row_scale = true;
    a->has_offset = true;
    a->v_ones = false;
    *out = a.release();
    return SB_OK;
}

extern "C" int sb_normalize(sb_mat *mat, int norm, const uint32_t *size_factors, sb_nmat **out) {
    if (!mat || !out) return sb_fail(SB_ERR_INVALID_ARG, "sb_normalize: NULL argument");
    SB_ENTER(mat->ctx);
    *out = nullptr;
    switch (norm) {
    case SB_NORM_CELLRANGER:  // normalization.rs:53, :84
        return sb_log_normalize(mat, 0, 0.0, SB_LOG_TWO, nullptr, 1, nullptr, out);
    case SB_NORM_CELLRANGER8: {  // :54-58, :85-89: scale_and_center(Axis(1), Some(ones))
        std::vector<double> ones(mat->m, 1.0);
        return sb_log_normalize(mat, 0, 0.0, SB_LOG_TWO, nullptr, 2, ones.data(), out);
    }
    case SB_NORM_SEURATLOG:  // :59, :90-92
        return sb_log_normalize(mat, 1, 10000.0, SB_LOG_E, nullptr, 1, nullptr, out);
    case SB_NORM_WITH_SIZE_FACTORS: {  // :93-95 (size_factors == None falls back to the cell totals, :148-160)
        const int rc = sb_log_normalize(mat, 0, 0.0, SB_LOG_TWO, size_factors, 1, nullptr, out);
        if (rc == SB_OK) (*out)->like_ok = false;  // a size-factor map: sb_normalize_like does not apply it
        return rc;
    }
    case SB_NORM_LOG_TRANSFORM: {  // :96-100
        std::vector<u32> ones(mat->n, 1u);
        return sb_log_normalize(mat, 1, 1.0, SB_LOG_TWO, ones.data(), 1, nullptr, out);
    }
    case SB_NORM_BINOMIAL_DEVIANCE:
        return normalize_binomial(mat, 1, out);
    case SB_NORM_BINOMIAL_PEARSON:
        return normalize_binomial(mat, 0, out);
    default:
        return sb_fail(SB_ERR_INVALID_ARG, "sb_normalize: not implemented (normalization %d)", norm);
    }
}

// the reference's map applied to the query's cells: col_scale = target / total_c from the query's own totals and its own L_c tables;
// log base, 1/sd row scales, the -mean/sd offset and the flags copied device to device (the m-vectors are the same on every rank)
extern "C" int sb_normalize_like(sb_mat *query, const sb_nmat *reference, sb_nmat **out) {
    if (!query || !reference || !out) return sb_fail(SB_ERR_INVALID_ARG, "sb_normalize_like: NULL argument");
    *out = nullptr;
    if (query->ctx != reference->ctx) return sb_fail(SB_ERR_INVALID_ARG, "sb_normalize_like: the query and the reference have different contexts");
    if (!reference->like_ok)
        return sb_fail(SB_ERR_UNSUPPORTED, "sb_normalize_like: the reference must be a log-chain normalization without size factors "
                                           "(CellRanger, CellRanger8, SeuratLog or sb_log_normalize without size factors)");
    if (query->m != reference->mat->m)
        return sb_fail(SB_ERR_INVALID_ARG, "sb_normalize_like: the query has %u genes, the reference %u", query->m, reference->mat->m);
    sb_ctx *ctx = query->ctx;
    SB_ENTER(ctx);
    std::unique_ptr<sb_nmat> a(new sb_nmat());
    a->mat = query;
    a->ctx = ctx;
    a->kind = 1;
    a->log_base = reference->log_base;
    SB_TRY(mat_cell_totals_dev(query));
    SB_TRY(log_col_tables(a.get(), reference->target, nullptr));
    a->has_row_scale = reference->has_row_scale;
    a->has_offset = reference->has_offset;
    a->v_ones = reference->v_ones;
    const size_t mb = (size_t)query->m * sizeof(double);
    if (a->has_row_scale) {
        SB_TRY(a->row_scale.alloc(query->m));
        if (mb) SB_CUDA(cudaMemcpyAsync(a->row_scale.p, reference->row_scale.p, mb, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    if (a->has_offset) {
        SB_TRY(a->u.alloc(query->m));
        if (mb) SB_CUDA(cudaMemcpyAsync(a->u.p, reference->u.p, mb, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = a.release();
    return SB_OK;
}

extern "C" int sb_normalize_fixed_point(sb_mat *mat, int log_base, uint32_t base, uint32_t exponent, sb_nmat **out) {
    if (!mat || !out) return sb_fail(SB_ERR_INVALID_ARG, "sb_normalize_fixed_point: NULL argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    // ones / (base.pow(exponent) as f64)  (normalization.rs:203-206): u32 pow, wrapping like release Rust
    u32 pw = 1;
    for (u32 i = 0; i < exponent; i++) pw *= base;
    double cs = 1.0 / (double)pw;
    // same as a log-normalize whose column scales are the constant `cs`: target = cs, size factors = 1
    std::vector<u32> ones(mat->n, 1u);
    return sb_log_normalize(mat, 1, cs, log_base, ones.data(), 1, nullptr, out);
}

extern "C" void sb_free_nmat(sb_nmat *a) {
    if (!a) return;
    cudaSetDevice(a->ctx->device);
    sb_set_alloc_stream(a->ctx->stream);
    cudaStreamSynchronize(a->ctx->stream);
    delete a;
}

extern "C" int sb_nmat_params(const sb_nmat *a, double *col_scale, double *row_scale, double *u, double *v) {
    if (!a) return sb_fail(SB_ERR_INVALID_ARG, "sb_nmat_params: NULL argument");
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    SB_ENTER(ctx);
    if (col_scale && mt->n) SB_CUDA(cudaMemcpyAsync(col_scale, a->col_scale.p, mt->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (row_scale) {
        if (a->has_row_scale) {
            if (mt->m) SB_CUDA(cudaMemcpyAsync(row_scale, a->row_scale.p, (size_t)mt->m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        } else
            for (u32 g = 0; g < mt->m; g++) row_scale[g] = 1.0;
    }
    if (u) {
        if (a->has_offset) {
            if (mt->m) SB_CUDA(cudaMemcpyAsync(u, a->u.p, (size_t)mt->m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        } else
            for (u32 g = 0; g < mt->m; g++) u[g] = 0.0;
    }
    if (v) {
        if (a->has_offset && !a->v_ones) {
            if (mt->n) SB_CUDA(cudaMemcpyAsync(v, a->v.p, mt->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        } else
            for (u64 c = 0; c < mt->n; c++) v[c] = a->has_offset ? 1.0 : 0.0;
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- host-facing products
static inline u32 even_up(u32 w) { return (w + 1) & ~1u; }

extern "C" int sb_nmat_dot(sb_nmat *a, const double *x, uint32_t w, double *out) {
    if (!a || !x || !out || w == 0) return sb_fail(SB_ERR_INVALID_ARG, "sb_nmat_dot: bad argument");
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    SB_ENTER(ctx);
    u32 ld = even_up(w);
    DevBuf<double> X, P;
    SB_TRY(X.alloc((size_t)mt->n * ld));
    SB_TRY(P.alloc(((size_t)mt->m + 1) * ld));
    SB_CUDA(cudaMemsetAsync(X.p, 0, (size_t)(mt->n ? mt->n : 1) * ld * sizeof(double), ctx->stream));
    if (mt->n)
        SB_CUDA(cudaMemcpy2DAsync(X.p, ld * sizeof(double), x, w * sizeof(double), w * sizeof(double), mt->n, cudaMemcpyHostToDevice, ctx->stream));
    SB_TRY(spmm_n(a, X.p, ld, w, P.p, ld));
    if (mt->m)
        SB_CUDA(cudaMemcpy2DAsync(out, w * sizeof(double), P.p, ld * sizeof(double), w * sizeof(double), mt->m, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

extern "C" int sb_nmat_rdot(sb_nmat *a, const double *b, uint32_t w, double *out) {
    if (!a || !b || !out || w == 0) return sb_fail(SB_ERR_INVALID_ARG, "sb_nmat_rdot: bad argument");
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    SB_ENTER(ctx);
    u32 ld = even_up(w);
    // Y[g, j] = b[j, g]
    std::vector<double> hy((size_t)mt->m * ld, 0.0);
    for (u32 j = 0; j < w; j++)
        for (u32 g = 0; g < mt->m; g++) hy[(size_t)g * ld + j] = b[(size_t)j * mt->m + g];
    DevBuf<double> Y, T, uy;
    SB_TRY(Y.alloc(hy.size()));
    SB_TRY(T.alloc((size_t)mt->n * ld));
    SB_TRY(uy.alloc(ld));
    if (!hy.empty()) SB_CUDA(cudaMemcpyAsync(Y.p, hy.data(), hy.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemsetAsync(T.p, 0, (size_t)(mt->n ? mt->n : 1) * ld * sizeof(double), ctx->stream));
    SB_TRY(spmm_t(a, Y.p, ld, w, T.p, ld, uy.p));
    std::vector<double> ht((size_t)mt->n * ld);
    if (!ht.empty()) SB_CUDA(cudaMemcpyAsync(ht.data(), T.p, ht.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    for (u64 c = 0; c < mt->n; c++)
        for (u32 j = 0; j < w; j++) out[(size_t)j * mt->n + c] = ht[(size_t)c * ld + j];
    return SB_OK;
}

// LowRankOffset::to_dense (low_rank_offset.rs:55-57): A = A . I through the gather kernel, test sizes only
extern "C" int sb_nmat_to_dense(sb_nmat *a, double *out) {
    if (!a || !out) return sb_fail(SB_ERR_INVALID_ARG, "sb_nmat_to_dense: NULL argument");
    sb_mat *mt = a->mat;
    if ((u64)mt->m * mt->n > (1ull << 26)) return sb_fail(SB_ERR_UNSUPPORTED, "sb_nmat_to_dense: matrix too large (debug path)");
    u32 m = mt->m;
    if (m == 0 || mt->n == 0) return SB_OK;
    std::vector<double> eye((size_t)m * m, 0.0), res((size_t)m * mt->n);
    for (u32 g = 0; g < m; g++) eye[(size_t)g * m + g] = 1.0;
    // eye . A = A  (m x n_local), row-major
    SB_TRY(sb_nmat_rdot(a, eye.data(), m, res.data()));
    memcpy(out, res.data(), res.size() * sizeof(double));
    return SB_OK;
}
