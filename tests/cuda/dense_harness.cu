// dense_harness.cu -- test entry points into the library's own dense kernels (dense_own.cu), for tests/test_dense_own_gpu.py.
// syrk_tall, gemm_tall, chol_inv, qr_chol and topk_select are internal (hidden) functions of libscanb200.so.  This file is linked
// with the library's object files into a separate shared library (-Bsymbolic), which exports the wrappers below plus its own copy
// of the public C ABI: a context for these wrappers is created with this library's sb_init and is never handed to libscanb200.so.
//
// Every wrapper takes host arrays.  An input array is copied whole to the device and the kernel's operand starts `off` doubles
// into it (off = 1 gives a base that is not 16-byte aligned).  An output array is copied whole in (as the caller pre-filled it)
// and whole back out, so that pad columns and rows past the operand can be checked against sentinels.  Device flags are zeroed
// before the call and returned.  Copies run on the context's stream; every wrapper ends with a stream synchronisation.
#include "../../scan_rs_b200/csrc/common.cuh"

int syrk_tall(sb_ctx *ctx, const double *A, u64 rows, u32 w, u32 ld, double *G);
int gemm_tall(sb_ctx *ctx, const double *A, u64 rows, u32 w, u32 lda, const double *S, u32 k, u32 lds, double *Out, u32 ldo, bool s_upper);
int chol_inv(sb_ctx *ctx, double *G, u32 w, double shift_coef, double *Rinv, int *flag);
int qr_chol(sb_ctx *ctx, double *A, double *tmp, u64 rows, u32 w, u32 ld, double *Rinv_out, int *flag, u64 rows_global);
int topk_select(sb_ctx *ctx, const double *W, const double *ev, u32 wq, u32 k, double *Wsel, double *Wsc, double *S);

#define DH_API extern "C" __attribute__((visibility("default")))

namespace {
// a device copy of a host array, copied back on request
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
struct DevFlag {
    int *p = nullptr;
    ~DevFlag() {
        if (p) cudaFree(p);
    }
    int init(sb_ctx *ctx) {
        SB_CUDA(cudaMalloc((void **)&p, sizeof(int)));
        SB_CUDA(cudaMemsetAsync(p, 0, sizeof(int), ctx->stream));
        return SB_OK;
    }
    int down(sb_ctx *ctx, int *h) {
        SB_CUDA(cudaMemcpyAsync(h, p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        return SB_OK;
    }
};
int finish(sb_ctx *ctx) {
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}
}  // namespace

// G (w x w, column-major) = A^T A for A = a[a_off ..] (rows x w, row-major, ld)
DH_API int dh_syrk(sb_ctx *ctx, const double *a, size_t n_a, u32 a_off, u64 rows, u32 w, u32 ld, double *g) {
    SB_ENTER(ctx);
    Dev A, G;
    SB_TRY(A.up(ctx, a, n_a));
    SB_TRY(G.up(ctx, g, (size_t)w * w));
    SB_TRY(syrk_tall(ctx, A.p + a_off, rows, w, ld, G.p));
    SB_TRY(G.down(ctx, g));
    return finish(ctx);
}

// Out = A . S.  in_place: Out is A itself (o_off, n_o and the initial `out` are ignored; the whole of A comes back in `out`)
DH_API int dh_gemm(sb_ctx *ctx, const double *a, size_t n_a, u32 a_off, u64 rows, u32 w, u32 lda, const double *s, size_t n_s, u32 k, u32 lds,
                   double *out, size_t n_o, u32 o_off, u32 ldo, int s_upper, int in_place) {
    SB_ENTER(ctx);
    Dev A, S, O;
    SB_TRY(A.up(ctx, a, n_a));
    SB_TRY(S.up(ctx, s, n_s));
    double *dout;
    if (in_place) {
        dout = A.p + a_off;
    } else {
        SB_TRY(O.up(ctx, out, n_o));
        dout = O.p + o_off;
    }
    const int rc = gemm_tall(ctx, A.p + a_off, rows, w, lda, S.p, k, lds, dout, ldo, s_upper != 0);
    if (rc != SB_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    SB_TRY(in_place ? A.down(ctx, out) : O.down(ctx, out));
    return finish(ctx);
}

// G (w x w, column-major) in, R out in its upper triangle (the strict lower triangle is left as the kernels leave it); rinv (w x w)
DH_API int dh_chol_inv(sb_ctx *ctx, double *g, u32 w, double shift_coef, double *rinv, int *flag) {
    SB_ENTER(ctx);
    Dev G, R;
    DevFlag F;
    SB_TRY(G.up(ctx, g, (size_t)w * w));
    SB_TRY(R.up(ctx, rinv, (size_t)w * w));
    SB_TRY(F.init(ctx));
    SB_TRY(chol_inv(ctx, G.p, w, shift_coef, R.p, F.p));
    SB_TRY(G.down(ctx, g));
    SB_TRY(R.down(ctx, rinv));
    SB_TRY(F.down(ctx, flag));
    return finish(ctx);
}

// A = a[a_off ..] (rows x w, row-major, ld) is replaced by Q; the whole array comes back in `q`.  rinv (w x w) may be NULL.
DH_API int dh_qr_chol(sb_ctx *ctx, const double *a, size_t n_a, u32 a_off, u64 rows, u32 w, u32 ld, double *q, double *rinv, int *flag,
                      u64 rows_global) {
    SB_ENTER(ctx);
    Dev A, T, R;
    DevFlag F;
    SB_TRY(A.up(ctx, a, n_a));
    SB_TRY(T.up(ctx, a, n_a));
    if (rinv) SB_TRY(R.up(ctx, rinv, (size_t)w * w));
    SB_TRY(F.init(ctx));
    SB_TRY(qr_chol(ctx, A.p + a_off, T.p + a_off, rows, w, ld, rinv ? R.p : nullptr, F.p, rows_global));
    SB_TRY(A.down(ctx, q));
    if (rinv) SB_TRY(R.down(ctx, rinv));
    SB_TRY(F.down(ctx, flag));
    return finish(ctx);
}

// W (wq x wq, column-major eigenvectors), ev (wq, ascending) -> wsel, wsc (wq x k, column-major), s (k)
DH_API int dh_topk(sb_ctx *ctx, const double *wv, const double *ev, u32 wq, u32 k, double *wsel, double *wsc, double *s) {
    SB_ENTER(ctx);
    Dev W, E, Ws, Wc, S;
    SB_TRY(W.up(ctx, wv, (size_t)wq * wq));
    SB_TRY(E.up(ctx, ev, wq));
    SB_TRY(Ws.up(ctx, wsel, (size_t)wq * k));
    SB_TRY(Wc.up(ctx, wsc, (size_t)wq * k));
    SB_TRY(S.up(ctx, s, k));
    SB_TRY(topk_select(ctx, W.p, E.p, wq, k, Ws.p, Wc.p, S.p));
    SB_TRY(Ws.down(ctx, wsel));
    SB_TRY(Wc.down(ctx, wsc));
    SB_TRY(S.down(ctx, s));
    return finish(ctx);
}
