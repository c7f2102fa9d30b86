// spmm_harness.cu -- test entry points into the library's sparse products (spmm.cu with the panelled gather of gather.cu and the
// bit-plane kernels of planes.cu), for tests/test_spmm_kernels_gpu.py.  spmm_t, spmm_n and nmat_moments are internal (hidden)
// functions of libscanb200.so.  This file is linked with the library's object files into a separate shared library (-Bsymbolic),
// which exports the wrappers below plus its own copy of the public C ABI: matrices for these wrappers are uploaded and normalized
// through this library's sb_* functions on a context created by its own sb_init, and never handed to libscanb200.so.
//
// The product wrappers take host arrays.  The operand array is copied whole to the device and the operand starts `off` doubles into
// it; the output array is copied whole in (as the caller pre-filled it) and whole back out, so that the columns and rows around the
// output block can be checked against sentinels.  Copies run on the context's stream; every wrapper ends with a stream
// synchronisation.
#include "../../scan_rs_b200/csrc/common.cuh"

int spmm_t(sb_nmat *a, const double *Y, u32 ldy, u32 w, double *out, u32 ldo, double *uy_scratch);
int spmm_n(sb_nmat *a, const double *X, u32 ldx, u32 w, double *P, u32 ldp);
int nmat_moments(sb_nmat *a, double *S);

#define SH_API extern "C" __attribute__((visibility("default")))

namespace {
struct Dev {
    double *p = nullptr;
    size_t n = 0;
    ~Dev() {
        if (p) cudaFree(p);
    }
    int up(sb_ctx *ctx, const double *h, size_t count) {
        n = count;
        SB_CUDA(cudaMalloc((void **)&p, (n ? n : 1) * sizeof(double)));
        if (n) SB_CUDA(cudaMemcpyAsync(p, h, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        return SB_OK;
    }
    int down(sb_ctx *ctx, double *h) {
        if (n) SB_CUDA(cudaMemcpyAsync(h, p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        return SB_OK;
    }
};
int finish(sb_ctx *ctx) {
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}
// a product that failed has enqueued nothing more: drain the copies and hand its status code back
int failed(sb_ctx *ctx, int rc) {
    cudaStreamSynchronize(ctx->stream);
    return rc;
}
}  // namespace

// T (n x w, ld ldo) = A^T . Y for Y = y[y_off ..] (m x w, ld ldy), T = out[o_off ..]
SH_API int sh_spmm_t(sb_nmat *a, const double *y, size_t n_y, u32 y_off, u32 ldy, u32 w, double *out, size_t n_o, u32 o_off, u32 ldo) {
    if (!a) return sb_fail(SB_ERR_INVALID_ARG, "sh_spmm_t: NULL matrix");
    sb_ctx *ctx = a->ctx;
    SB_ENTER(ctx);
    Dev Y, O, uy;
    SB_TRY(Y.up(ctx, y, n_y));
    SB_TRY(O.up(ctx, out, n_o));
    SB_CUDA(cudaMalloc((void **)&uy.p, ((size_t)w + 2) * sizeof(double)));
    const int rc = spmm_t(a, Y.p + y_off, ldy, w, O.p + o_off, ldo, uy.p);
    if (rc != SB_OK) return failed(ctx, rc);
    SB_TRY(O.down(ctx, out));
    return finish(ctx);
}

// P (m x w, ld ldp, plus the row m the product uses for v^T X) = A . X for X = x[x_off ..] (n x w, ld ldx), P = out[o_off ..]
SH_API int sh_spmm_n(sb_nmat *a, const double *x, size_t n_x, u32 x_off, u32 ldx, u32 w, double *out, size_t n_o, u32 o_off, u32 ldp) {
    if (!a) return sb_fail(SB_ERR_INVALID_ARG, "sh_spmm_n: NULL matrix");
    sb_ctx *ctx = a->ctx;
    SB_ENTER(ctx);
    Dev X, O;
    SB_TRY(X.up(ctx, x, n_x));
    SB_TRY(O.up(ctx, out, n_o));
    const int rc = spmm_n(a, X.p + x_off, ldx, w, O.p + o_off, ldp);
    if (rc != SB_OK) return failed(ctx, rc);
    SB_TRY(O.down(ctx, out));
    return finish(ctx);
}

// The layout the products run on.  info[0] planes active, [1] L, [2 .. 8) G_1 .. G_6, [8] T-side units, [9] N-side units,
// [10] T-side work items, [11] N-side work items, [12] gd (ranks of the dense half), [13] calibration rounds of the T-side gather,
// [14] cold (sparse) entries, [15] all entries (both capped at 2^32 - 1).  hot_idx (capacity m): the gene of every rank < G_1.
SH_API int sh_plane_layout(sb_nmat *a, u32 *info, u32 *hot_idx) {
    if (!a || !info) return sb_fail(SB_ERR_INVALID_ARG, "sh_plane_layout: NULL argument");
    const sb_mat *mt = a->mat;
    sb_ctx *ctx = a->ctx;
    SB_ENTER(ctx);
    const PlaneSet &pl = mt->pl;
    info[0] = pl.active ? 1u : 0u;
    info[1] = pl.L;
    for (u32 k = 0; k < PL_MAX_LEVELS; k++) info[2 + k] = pl.G[k];
    info[8] = pl.n_units_t;
    info[9] = pl.n_units_n;
    info[10] = pl.n_items_t;
    info[11] = pl.n_items_n;
    info[12] = mt->gd;
    info[13] = (u32)mt->t_calibrated;
    const bool hybrid = mt->gd > 0;
    info[14] = (u32)std::min<u64>(hybrid ? mt->cold_nnz : mt->nnz, 0xFFFFFFFFull);
    info[15] = (u32)std::min<u64>(mt->nnz, 0xFFFFFFFFull);
    if (hot_idx && pl.active && pl.G[0]) SB_CUDA(cudaMemcpyAsync(hot_idx, mt->hot_idx.p, (size_t)pl.G[0] * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    return finish(ctx);
}

// The per-gene moments of a log-normalized matrix (K5): S1[g] = sum_c L_gc, S2[g] = sum_c L_gc^2 over the stored entries, sparse
// kernel over the cold entries plus the plane kernels' moment mode over the rest
SH_API int sh_gene_moments(sb_nmat *a, double *s1, double *s2) {
    if (!a || !s1 || !s2) return sb_fail(SB_ERR_INVALID_ARG, "sh_gene_moments: NULL argument");
    if (a->kind != 1) return sb_fail(SB_ERR_UNSUPPORTED, "sh_gene_moments: log-chain normalizations only");
    sb_ctx *ctx = a->ctx;
    SB_ENTER(ctx);
    const u32 m = a->mat->m;
    DevBuf<double> S;
    SB_TRY(S.alloc(2 * (size_t)m + 1));
    SB_TRY(nmat_moments(a, S.p));
    if (m) {
        SB_CUDA(cudaMemcpyAsync(s1, S.p, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(s2, S.p + m, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    return finish(ctx);
}
