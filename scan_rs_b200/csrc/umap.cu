// umap.cu -- the UMAP embedding of the kNN lists (the reference workspace's `umap-rs`, a port of umap-learn): the fuzzy kNN graph
// and an epoch-synchronous, bit-reproducible layout.  The rules are stated beside the entry points in include/scanb200.h and
// restated by oracle/umap.py.
//
//   graph    k_um_dist: a thread per (row, slot) validates the slot and computes its distance; k_um_smooth: a thread per row finds
//            rho and runs umap-learn's sigma bisection; k_um_member: the memberships.  The union sorts the forward pair keys and
//            the transposed ones (the value names the source slot, the top bit tags a transposed entry), k_um_combine joins the
//            (up to two) entries of a pair, and a flagged select keeps the non-zero weights: a symmetric CSR, columns ascending.
//   layout   prune + schedule on the directed edges, then per epoch k_um_epoch (a thread per edge: attractive update of both
//            ends, the head's negative samples) and k_um_apply.  Every epoch reads one snapshot of the positions; each
//            contribution alpha grad is rounded to an integer multiple of 2^-32 and summed per vertex with 64-bit atomics, so the
//            sums do not depend on the order the atomics land in, and the positions are kept as those integers.  No host round
//            trip inside the epoch loop.
//   transform  new points into a fixed embedding (umap-learn's transform): the graph from the fit's kernels against a second
//            point set with rho = 0, then k_ut_start and k_ut_layout, a thread per query row running every epoch in one launch.
#include <cmath>

#include <cub/cub.cuh>

#include "common.cuh"

#define UM_PAD 0xFFFFFFFFu
#define UM_MAX_K 128
#define UM_MAX_COMPONENTS 8
#define UM_FIX 4294967296.0        // positions and contributions are integers in units of 2^-32
#define UM_IFIX (1.0 / 4294967296.0)
#define UM_TAG (1ull << 63)
#define UM_INIT_LIMIT 1073741824.0  // |user start| < 2^30: its fixed-point value fits an i64 with room to move

typedef unsigned long long ull;
typedef long long i64;

static int um_grid(sb_ctx *ctx, u64 items, int per_block) {
    return (int)std::max<u64>(1, std::min<u64>((items + per_block - 1) / per_block, (u64)ctx->sm_count * 32));
}

// ---------------------------------------------------------------- graph
__global__ void k_um_dist(const double *__restrict__ X, const double *__restrict__ P, u64 np, const u32 *__restrict__ nbr, u64 n, u32 dim,
                          u32 k, int full, double *__restrict__ d, int *__restrict__ err) {
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < n * k; s += (u64)gridDim.x * blockDim.x) {
        const u64 i = s / k;
        const u32 t = (u32)(s - i * k), j = nbr[s];
        double r = 0.0;
        int e = 0;
        if (j != UM_PAD) {
            if (t && nbr[s - 1] == UM_PAD) e |= 8;
            if (j >= np) e |= 1;
            else if (!full && j == i) e |= 2;
            for (u32 q = 0; q < t; q++)
                if (nbr[i * k + q] == j) e |= 4;
            if (!e) {
                const double *xi = X + i * dim, *xj = P + (u64)j * dim;
                for (u32 c = 0; c < dim; c++) {
                    const double df = __dsub_rn(xj[c], xi[c]);
                    r = __dadd_rn(r, __dmul_rn(df, df));
                }
                r = sqrt(r);
            }
        } else if (full) {
            e |= 16;
        }
        d[s] = r;
        if (e) atomicOr(err, e);
    }
}

// thread per row: rho, the row sum of the distances, sigma by umap-learn's bisection with the row-mean floor (rows with rho = 0
// get the global floor later: flag[0] = 1), cnt[0] += listed entries + 1.  rho0 = 1 (the transform's local connectivity 0): rho = 0
// on every row and cnt[0] += listed entries
__global__ void k_um_smooth(const double *__restrict__ d, const u32 *__restrict__ nbr, u64 n, u32 k, double target, int rho0,
                            double *__restrict__ rho, double *__restrict__ sigma, double *__restrict__ rowsum, int *__restrict__ flag,
                            ull *__restrict__ cnt) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const double *di = d + i * k;
        const u32 *ri = nbr + i * k;
        u32 m = 0;
        double r = INFINITY, s = 0.0;
        for (u32 t = 0; t < k; t++) {
            if (ri[t] == UM_PAD) continue;
            m++;
            s = __dadd_rn(s, di[t]);
            if (!rho0 && di[t] > 0.0 && di[t] < r) r = di[t];
        }
        if (r == INFINITY) r = 0.0;
        double lo = 0.0, hi = INFINITY, mid = 1.0;
        for (int it = 0; it < 64; it++) {
            double psum = 0.0;
            for (u32 t = 0; t < k; t++) {
                if (ri[t] == UM_PAD) continue;
                const double x = __dsub_rn(di[t], r);
                psum = __dadd_rn(psum, x > 0.0 ? exp(-__ddiv_rn(x, mid)) : 1.0);
            }
            if (fabs(__dsub_rn(psum, target)) < 1e-5) break;
            if (psum > target) {
                hi = mid;
                mid = __ddiv_rn(__dadd_rn(lo, hi), 2.0);
            } else {
                lo = mid;
                mid = isinf(hi) ? __dmul_rn(mid, 2.0) : __ddiv_rn(__dadd_rn(lo, hi), 2.0);
            }
        }
        if (r > 0.0) {
            const double fl = __dmul_rn(1e-3, __ddiv_rn(s, (double)(m + 1)));
            if (mid < fl) mid = fl;
        } else {
            atomicOr(flag, 1);
        }
        rho[i] = r;
        sigma[i] = mid;
        rowsum[i] = s;
        atomicAdd(cnt, (ull)(rho0 ? m : m + 1));
    }
}

__global__ void k_um_global_floor(const double *__restrict__ rho, double *__restrict__ sigma, u64 n, double fl) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (!(rho[i] > 0.0) && sigma[i] < fl) sigma[i] = fl;
}

// thread per (row, slot): w = exp(-max(0, d - rho) / sigma); the forward key (i << 32 | j, value: the slot) and the transposed key
// (j << 32 | i, value: the slot | UM_TAG); all-ones keys at padding.  keys = NULL: the weights only
__global__ void k_um_member(const double *__restrict__ d, const u32 *__restrict__ nbr, u64 n, u32 k, const double *__restrict__ rho,
                            const double *__restrict__ sigma, double *__restrict__ w, u64 *__restrict__ keys, u64 *__restrict__ vals) {
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < n * k; s += (u64)gridDim.x * blockDim.x) {
        const u64 i = s / k;
        const u32 j = nbr[s];
        if (j == UM_PAD) {
            w[s] = 0.0;
            if (!keys) continue;
            keys[2 * s] = keys[2 * s + 1] = ~0ull;
            vals[2 * s] = vals[2 * s + 1] = 0;
            continue;
        }
        const double x = __dsub_rn(d[s], rho[i]);
        w[s] = x > 0.0 ? exp(-__ddiv_rn(x, sigma[i])) : 1.0;
        if (!keys) continue;
        keys[2 * s] = (i << 32) | j;
        vals[2 * s] = s;
        keys[2 * s + 1] = ((u64)j << 32) | i;
        vals[2 * s + 1] = s | UM_TAG;
    }
}

// thread per sorted entry: the first entry of a pair joins a = w_ij and b = w_ji into mix (a + b - a b) + (1 - mix) a b
__global__ void k_um_combine(const u64 *__restrict__ keys, const u64 *__restrict__ vals, u64 count, const double *__restrict__ w, double mix,
                             double one_minus_mix, double *__restrict__ out, char *__restrict__ keep) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (u64)gridDim.x * blockDim.x) {
        keep[x] = 0;
        out[x] = 0.0;
        if (x && keys[x] == keys[x - 1]) continue;
        double a = 0.0, b = 0.0;
        for (u64 y = x; y < count && y < x + 2 && keys[y] == keys[x]; y++) {
            const u64 v = vals[y];
            if (v & UM_TAG) b = w[v & ~UM_TAG];
            else a = w[v];
        }
        const double p = __dmul_rn(a, b);
        const double r = __dadd_rn(__dmul_rn(mix, __dsub_rn(__dadd_rn(a, b), p)), __dmul_rn(one_minus_mix, p));
        out[x] = r;
        keep[x] = r > 0.0;
    }
}

// first position with keys[pos] >= (r << 32), for every row r in [0, n]; and the column of every entry
__global__ void k_um_rows(const u64 *__restrict__ keys, u64 nnz, u64 n, u64 *__restrict__ ptr) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r <= n; r += (u64)gridDim.x * blockDim.x) {
        const u64 want = r << 32;
        u64 lo = 0, hi = nnz;
        while (lo < hi) {
            const u64 mid = (lo + hi) >> 1;
            if (keys[mid] < want) lo = mid + 1;
            else hi = mid;
        }
        ptr[r] = lo;
    }
}
__global__ void k_um_cols(const u64 *__restrict__ keys, u64 nnz, u32 *__restrict__ idx) {
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (u64)gridDim.x * blockDim.x) idx[e] = (u32)keys[e];
}

template <typename T>
int um_select(sb_ctx *ctx, const T *in, const char *flags, T *out, u64 count, u64 *d_num) {
    size_t tb = 0;
    SB_CUDA(cub::DeviceSelect::Flagged(nullptr, tb, in, flags, out, d_num, count, ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tb));
    SB_CUDA(cub::DeviceSelect::Flagged(tmp.p, tb, in, flags, out, d_num, count, ctx->stream));
    count_launch(ctx, false);
    return SB_OK;
}
template int um_select<u32>(sb_ctx *, const u32 *, const char *, u32 *, u64, u64 *);
template int um_select<u64>(sb_ctx *, const u64 *, const char *, u64 *, u64, u64 *);
template int um_select<double>(sb_ctx *, const double *, const char *, double *, u64, u64 *);

// keys (row << 32 | col, ascending) of nnz entries -> g.ptr, g.idx
int um_rows_from_keys(sb_ctx *ctx, const u64 *keys, UmGraph &g) {
    SB_TRY(g.ptr.alloc(g.n + 1));
    SB_TRY(g.idx.alloc(g.nnz));
    k_um_rows<<<um_grid(ctx, g.n + 1, 256), 256, 0, ctx->stream>>>(keys, g.nnz, g.n, g.ptr.p);
    count_launch(ctx);
    if (g.nnz) {
        k_um_cols<<<um_grid(ctx, g.nnz, 256), 256, 0, ctx->stream>>>(keys, g.nnz, g.idx.p);
        count_launch(ctx);
    }
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

// X [n x dim], nbr [n x k] on the device -> g, rho, sigma (device)
static int um_graph_build(sb_ctx *ctx, const double *X, const u32 *nbr, u64 n, u32 dim, u32 k, double mix, UmGraph &g, DevBuf<double> &rho,
                          DevBuf<double> &sigma, const char *fn) {
    TraceScope tr(ctx, "umap: fuzzy graph");
    const u64 nk = n * k;
    DevBuf<double> d, rs, w;
    DevBuf<int> flags;  // [0] error bits, [1] a row with rho = 0
    DevBuf<ull> cnt;
    SB_TRY(d.alloc(nk));
    SB_TRY(rs.alloc(n));
    SB_TRY(w.alloc(nk));
    SB_TRY(rho.alloc(n));
    SB_TRY(sigma.alloc(n));
    SB_TRY(flags.alloc(2));
    SB_TRY(cnt.alloc(1));
    SB_CUDA(cudaMemsetAsync(flags.p, 0, 2 * sizeof(int), ctx->stream));
    SB_CUDA(cudaMemsetAsync(cnt.p, 0, sizeof(ull), ctx->stream));
    g.n = n;
    if (n) {
        k_um_dist<<<um_grid(ctx, nk, 256), 256, 0, ctx->stream>>>(X, X, n, nbr, n, dim, k, 0, d.p, flags.p);
        k_um_smooth<<<um_grid(ctx, n, 128), 128, 0, ctx->stream>>>(d.p, nbr, n, k, std::log2((double)k + 1.0), 0, rho.p, sigma.p, rs.p, flags.p + 1,
                                                                   cnt.p);
        count_launch(ctx);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
    }
    int hf[2];
    ull hc = 0;
    SB_CUDA(cudaMemcpyAsync(hf, flags.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(&hc, cnt.p, sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (hf[0])
        return sb_fail(SB_ERR_INVALID_ARG, "%s: invalid neighbour lists:%s%s%s%s", fn, hf[0] & 1 ? " an index >= n" : "", hf[0] & 2 ? " a self index" : "",
                       hf[0] & 4 ? " a duplicate in a row" : "", hf[0] & 8 ? " padding before the row end" : "");
    if (hf[1]) {  // the global mean distance, summed row by row in order
        std::vector<double> h(n);
        SB_CUDA(cudaMemcpyAsync(h.data(), rs.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        double tot = 0.0;
        for (u64 i = 0; i < n; i++) tot += h[i];
        k_um_global_floor<<<um_grid(ctx, n, 256), 256, 0, ctx->stream>>>(rho.p, sigma.p, n, 1e-3 * (tot / (double)hc));
        count_launch(ctx);
    }
    TraceScope tru(ctx, "umap: fuzzy union");
    const u64 listed = hc - n, np = 2 * nk;  // the valid keys sort first; the all-ones keys of padding last
    DevBuf<u64> keys, vals;
    SB_TRY(keys.alloc(np));
    SB_TRY(vals.alloc(np));
    if (n) {
        k_um_member<<<um_grid(ctx, nk, 256), 256, 0, ctx->stream>>>(d.p, nbr, n, k, rho.p, sigma.p, w.p, keys.p, vals.p);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
    }
    d.release();
    const u64 cnt2 = 2 * listed;
    DevBuf<double> comb, gw;
    DevBuf<char> keep;
    DevBuf<u64> gk, num;
    SB_TRY(comb.alloc(cnt2));
    SB_TRY(keep.alloc(cnt2));
    SB_TRY(gk.alloc(cnt2));
    SB_TRY(gw.alloc(cnt2));
    SB_TRY(num.alloc(1));
    u64 nnz = 0;
    if (cnt2) {
        SB_TRY(sort_pairs(ctx, keys, vals, np));
        k_um_combine<<<um_grid(ctx, cnt2, 256), 256, 0, ctx->stream>>>(keys.p, vals.p, cnt2, w.p, mix, 1.0 - mix, comb.p, keep.p);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
        SB_TRY(um_select(ctx, keys.p, keep.p, gk.p, cnt2, num.p));
        SB_TRY(um_select(ctx, comb.p, keep.p, gw.p, cnt2, num.p));
        SB_CUDA(cudaMemcpyAsync(&nnz, num.p, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    g.nnz = nnz;
    SB_TRY(um_rows_from_keys(ctx, gk.p, g));
    g.w.swap(gw);
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- layout
// warp per row: every entry's head (the row), the max weight (positive doubles order as their bits) and the max degree
__global__ void k_um_heads(const u64 *__restrict__ ptr, const double *__restrict__ w, u64 n, u32 *__restrict__ head, ull *__restrict__ mx) {
    const int lane = threadIdx.x & 31;
    for (u64 i = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += ((u64)gridDim.x * blockDim.x) >> 5) {
        ull m = 0;
        for (u64 x = ptr[i] + lane; x < ptr[i + 1]; x += 32) {
            head[x] = (u32)i;
            const ull v = (ull)__double_as_longlong(w[x]);
            m = v > m ? v : m;
        }
        for (int o = 16; o > 0; o >>= 1) {
            const ull v = __shfl_xor_sync(0xffffffffu, m, o);
            m = v > m ? v : m;
        }
        if (lane == 0) {
            if (m) atomicMax(&mx[0], m);
            atomicMax(&mx[1], (ull)(ptr[i + 1] - ptr[i]));
        }
    }
}
__global__ void k_um_prune(const double *__restrict__ w, u64 nnz, double thr, char *__restrict__ keep) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < nnz; x += (u64)gridDim.x * blockDim.x) keep[x] = w[x] >= thr;
}
// epochs_per_sample = w_max / w, per negative sample / rate; the next epochs start at those values
__global__ void k_um_schedule(const double *__restrict__ w, u64 E, double wmax, double rate, double *__restrict__ eps, double *__restrict__ epn,
                              double *__restrict__ ens, double *__restrict__ enn) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < E; x += (u64)gridDim.x * blockDim.x) {
        const double s = __ddiv_rn(wmax, w[x]), q = rate > 0.0 ? __ddiv_rn(s, rate) : INFINITY;
        eps[x] = ens[x] = s;
        epn[x] = enn[x] = q;
    }
}

struct EpochArgs {
    const u32 *head, *tail;
    const double *eps, *epn;
    double *ens, *enn;
    const i64 *Y;  // [n x NC] positions, units of 2^-32
    ull *acc;      // [n x NC] this epoch's sums
    u64 E, n;
    double a, b, bm1, m2ab, two_gb, alpha, epoch;
    u64 key;       // mix64(mix64(seed) ^ epoch)
    int negatives;
};

__device__ __forceinline__ double um_clip(double g) { return g > 4.0 ? 4.0 : (g < -4.0 ? -4.0 : g); }
__device__ __forceinline__ i64 um_fix(double g, double alpha) { return __double2ll_rn(__dmul_rn(__dmul_rn(g, alpha), UM_FIX)); }

// thread per directed edge of the pruned graph
template <int NC>
__global__ void __launch_bounds__(256) k_um_epoch(EpochArgs p) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < p.E; x += (u64)gridDim.x * blockDim.x) {
        const double ns = p.ens[x];
        if (ns > p.epoch) continue;
        const u32 j = p.head[x], k = p.tail[x];
        double yj[NC], yk[NC];
        i64 h[NC];
        double d2 = 0.0;
#pragma unroll
        for (int c = 0; c < NC; c++) {
            yj[c] = __dmul_rn((double)p.Y[(u64)j * NC + c], UM_IFIX);
            yk[c] = __dmul_rn((double)p.Y[(u64)k * NC + c], UM_IFIX);
            const double df = __dsub_rn(yj[c], yk[c]);
            d2 = __dadd_rn(d2, __dmul_rn(df, df));
        }
        const double gc = d2 > 0.0 ? __ddiv_rn(__dmul_rn(p.m2ab, pow(d2, p.bm1)), __dadd_rn(__dmul_rn(p.a, pow(d2, p.b)), 1.0)) : 0.0;
#pragma unroll
        for (int c = 0; c < NC; c++) {
            h[c] = um_fix(um_clip(__dmul_rn(gc, __dsub_rn(yj[c], yk[c]))), p.alpha);
            if (h[c]) atomicAdd(&p.acc[(u64)k * NC + c], (ull)(-h[c]));
        }
        p.ens[x] = __dadd_rn(ns, p.eps[x]);
        if (p.negatives) {
            const double epn = p.epn[x], nn_f = p.enn[x];
            i64 nn = (i64)__ddiv_rn(__dsub_rn(p.epoch, nn_f), epn);
            if (nn < 0) nn = 0;
            const u64 k2 = um_mix64(p.key ^ x);
            for (i64 s = 0; s < nn; s++) {
                const u64 v = um_mix64(k2 ^ (u64)s) % p.n;
                if (v == j) continue;
                double dd = 0.0;
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    yk[c] = __dmul_rn((double)p.Y[v * NC + c], UM_IFIX);
                    const double df = __dsub_rn(yj[c], yk[c]);
                    dd = __dadd_rn(dd, __dmul_rn(df, df));
                }
                if (dd > 0.0) {
                    const double g = __ddiv_rn(p.two_gb, __dmul_rn(__dadd_rn(0.001, dd), __dadd_rn(__dmul_rn(p.a, pow(dd, p.b)), 1.0)));
#pragma unroll
                    for (int c = 0; c < NC; c++) h[c] += um_fix(um_clip(__dmul_rn(g, __dsub_rn(yj[c], yk[c]))), p.alpha);
                } else {
                    const i64 f = um_fix(4.0, p.alpha);
#pragma unroll
                    for (int c = 0; c < NC; c++) h[c] += f;
                }
            }
            p.enn[x] = __dadd_rn(nn_f, __dmul_rn((double)nn, epn));
        }
#pragma unroll
        for (int c = 0; c < NC; c++)
            if (h[c]) atomicAdd(&p.acc[(u64)j * NC + c], (ull)h[c]);
    }
}

__global__ void k_um_apply(i64 *__restrict__ Y, ull *__restrict__ acc, u64 count) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (u64)gridDim.x * blockDim.x) {
        Y[x] = (i64)((ull)Y[x] + acc[x]);
        acc[x] = 0;
    }
}

template <int NC>
static void um_launch_epoch(sb_ctx *ctx, const EpochArgs &a) {
    k_um_epoch<NC><<<um_grid(ctx, a.E, 256), 256, 0, ctx->stream>>>(a);
}

// ---------------------------------------------------------------- start positions
// block per column c < nc of A [n x ld]: lo[c], hi[c]
__global__ void k_um_col_range(const double *__restrict__ A, u64 n, u32 ld, double *__restrict__ lo, double *__restrict__ hi) {
    __shared__ double sl[32], sh[32];
    const u32 c = blockIdx.x;
    double l = INFINITY, h = -INFINITY;
    for (u64 i = threadIdx.x; i < n; i += blockDim.x) {
        const double v = A[i * ld + c];
        l = fmin(l, v);
        h = fmax(h, v);
    }
    for (int o = 16; o > 0; o >>= 1) {
        l = fmin(l, __shfl_xor_sync(0xffffffffu, l, o));
        h = fmax(h, __shfl_xor_sync(0xffffffffu, h, o));
    }
    if ((threadIdx.x & 31) == 0) {
        sl[threadIdx.x >> 5] = l;
        sh[threadIdx.x >> 5] = h;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (u32 w = 1; w < blockDim.x >> 5; w++) {
            l = fmin(l, sl[w]);
            h = fmax(h, sh[w]);
        }
        lo[c] = l;
        hi[c] = h;
    }
}
// mode 0: 10 (a - lo) / (hi - lo) per column (0 for a constant column); 1: the counter hash, uniform [-10, 10); 2: a as given
__global__ void k_um_init(const double *__restrict__ A, u64 n, u32 ld, u32 nc, int mode, const double *__restrict__ lo, const double *__restrict__ hi,
                          u64 key, i64 *__restrict__ Y) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < n * nc; x += (u64)gridDim.x * blockDim.x) {
        const u64 i = x / nc;
        const u32 c = (u32)(x - i * nc);
        double v;
        if (mode == 0) v = hi[c] > lo[c] ? __ddiv_rn(__dmul_rn(10.0, __dsub_rn(A[i * ld + c], lo[c])), __dsub_rn(hi[c], lo[c])) : 0.0;
        else if (mode == 1) v = __dadd_rn(-10.0, __dmul_rn(20.0, __dmul_rn((double)(um_mix64(key ^ x) >> 11), 0x1p-53)));
        else v = A[i * ld + c];
        Y[x] = __double2ll_rn(__dmul_rn(v, UM_FIX));
    }
}

// ---------------------------------------------------------------- options
struct UmOpts {
    u32 nc, n_epochs, rate, init;
    double min_dist, spread, a, b, lr, gamma, mix;
    u64 seed;
};

static int um_opts(const sb_umap_opts *o, UmOpts &out, const char *fn) {
    out = UmOpts{2, 0, 5, SB_UMAP_INIT_PCA, 0.1, 1.0, 0.0, 0.0, 1.0, 1.0, 1.0, 0};
    if (!o) return SB_OK;
    out = UmOpts{o->n_components, o->n_epochs, o->negative_sample_rate, o->init, o->min_dist, o->spread, o->a, o->b, o->learning_rate,
                 o->repulsion_strength, o->set_op_mix_ratio, o->seed};
    if (out.nc < 1 || out.nc > UM_MAX_COMPONENTS) return sb_fail(SB_ERR_INVALID_ARG, "%s: n_components must be 1..%d", fn, UM_MAX_COMPONENTS);
    if (!(out.spread > 0.0) || !std::isfinite(out.spread)) return sb_fail(SB_ERR_INVALID_ARG, "%s: spread must be finite and > 0", fn);
    if (!(out.min_dist >= 0.0) || !(out.min_dist <= out.spread)) return sb_fail(SB_ERR_INVALID_ARG, "%s: min_dist must be in [0, spread]", fn);
    const bool fit = out.a == 0.0 && out.b == 0.0, given = out.a > 0.0 && out.b > 0.0 && std::isfinite(out.a) && std::isfinite(out.b);
    if (!fit && !given) return sb_fail(SB_ERR_INVALID_ARG, "%s: a and b must both be 0 (fit) or both finite and > 0", fn);
    if (!(out.lr > 0.0) || !std::isfinite(out.lr)) return sb_fail(SB_ERR_INVALID_ARG, "%s: learning_rate must be finite and > 0", fn);
    if (!(out.gamma >= 0.0) || !std::isfinite(out.gamma)) return sb_fail(SB_ERR_INVALID_ARG, "%s: repulsion_strength must be finite and >= 0", fn);
    if (!(out.mix >= 0.0 && out.mix <= 1.0)) return sb_fail(SB_ERR_INVALID_ARG, "%s: set_op_mix_ratio must be in [0, 1]", fn);
    if (out.init > SB_UMAP_INIT_USER) return sb_fail(SB_ERR_INVALID_ARG, "%s: init must be SB_UMAP_INIT_PCA, _RANDOM or _USER", fn);
    return SB_OK;
}

// least squares of 1 / (1 + a x^(2b)) to umap-learn's target on linspace(0, 3 spread, 300): Levenberg-Marquardt from (1, 1), as
// oracle/umap.py fit_ab states it
static void um_fit_ab(double spread, double min_dist, double &a_out, double &b_out) {
    const int N = 300;
    std::vector<double> x(N), y(N), lx(N), t(N), den(N), r(N), t2(N), den2(N), r2(N);
    const double stop = spread * 3.0, step = stop / (N - 1);
    for (int i = 0; i < N; i++) {
        x[i] = i == N - 1 ? stop : i * step;
        y[i] = x[i] < min_dist ? 1.0 : std::exp(-(x[i] - min_dist) / spread);
        lx[i] = x[i] > 0.0 ? std::log(x[i]) : 0.0;
    }
    auto model = [&](double a, double b, std::vector<double> &tt, std::vector<double> &dd, std::vector<double> &rr) {
        double c = 0.0;
        for (int i = 0; i < N; i++) {
            tt[i] = x[i] > 0.0 ? std::exp(2.0 * b * lx[i]) : 0.0;
            dd[i] = 1.0 + a * tt[i];
            rr[i] = 1.0 / dd[i] - y[i];
            c += rr[i] * rr[i];
        }
        return c;
    };
    double a = 1.0, b = 1.0, lam = 1e-3;
    double cost = model(a, b, t, den, r);
    for (int it = 0; it < 500; it++) {
        double haa = 0, hab = 0, hbb = 0, ga = 0, gb = 0;
        for (int i = 0; i < N; i++) {
            const double d2 = den[i] * den[i], ja = -t[i] / d2, jb = -(2.0 * a) * lx[i] * t[i] / d2;
            haa += ja * ja;
            hab += ja * jb;
            hbb += jb * jb;
            ga += ja * r[i];
            gb += jb * r[i];
        }
        bool done = true;
        while (lam < 1e16) {
            const double m00 = haa * (1.0 + lam), m11 = hbb * (1.0 + lam), det = m00 * m11 - hab * hab;
            const double da = (-ga * m11 + gb * hab) / det, db = (-gb * m00 + ga * hab) / det, na = a + da, nb = b + db;
            if (na > 0.0 && nb > 0.0) {
                const double c2 = model(na, nb, t2, den2, r2);
                if (c2 < cost) {
                    done = std::fabs(da) <= 1e-15 * std::fabs(a) && std::fabs(db) <= 1e-15 * std::fabs(b);
                    a = na;
                    b = nb;
                    t.swap(t2);
                    den.swap(den2);
                    r.swap(r2);
                    cost = c2;
                    lam /= 10.0;
                    break;
                }
            }
            lam *= 10.0;
        }
        if (done) break;
    }
    a_out = a;
    b_out = b;
}

// start positions from A [n x ld] (mode 0 scales its first nc columns, 2 takes them, 1 ignores A)
static int um_init(sb_ctx *ctx, const double *A, u64 n, u32 ld, const UmOpts &o, DevBuf<i64> &Y) {
    SB_TRY(Y.alloc(n * o.nc));
    DevBuf<double> lo, hi;
    SB_TRY(lo.alloc(o.nc));
    SB_TRY(hi.alloc(o.nc));
    const int mode = o.init == SB_UMAP_INIT_PCA ? 0 : o.init == SB_UMAP_INIT_RANDOM ? 1 : 2;
    if (n && mode == 0) {
        k_um_col_range<<<o.nc, 256, 0, ctx->stream>>>(A, n, ld, lo.p, hi.p);
        count_launch(ctx);
    }
    if (n) {
        k_um_init<<<um_grid(ctx, n * o.nc, 256), 256, 0, ctx->stream>>>(A, n, ld, o.nc, mode, lo.p, hi.p, um_mix64(um_mix64(o.seed) ^ ~0ull), Y.p);
        count_launch(ctx);
    }
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

// steps 4-6 on g (consumed) from the start Y -> Y
static int um_layout(sb_ctx *ctx, UmGraph &g, DevBuf<i64> &Y, const UmOpts &o, sb_umap_info *info, const char *fn) {
    const u64 n = g.n, nnz = g.nnz;
    double a = o.a, b = o.b;
    if (!(a > 0.0 && b > 0.0)) um_fit_ab(o.spread, o.min_dist, a, b);
    const u32 n_epochs = o.n_epochs ? o.n_epochs : (n <= 10000 ? 500 : 200);
    info->a = a;
    info->b = b;
    info->n_epochs = n_epochs;
    info->n_edges = nnz;
    info->n_edges_used = 0;
    info->max_weight = 0.0;
    if (!nnz) return SB_OK;
    TraceScope tr(ctx, "umap: schedule and epochs");
    DevBuf<u32> head, ph, pt;
    DevBuf<ull> mx;
    DevBuf<char> keep;
    DevBuf<double> pw;
    DevBuf<u64> num;
    SB_TRY(head.alloc(nnz));
    SB_TRY(mx.alloc(2));
    SB_TRY(keep.alloc(nnz));
    SB_TRY(ph.alloc(nnz));
    SB_TRY(pt.alloc(nnz));
    SB_TRY(pw.alloc(nnz));
    SB_TRY(num.alloc(1));
    SB_CUDA(cudaMemsetAsync(mx.p, 0, 2 * sizeof(ull), ctx->stream));
    k_um_heads<<<um_grid(ctx, n * 32, 256), 256, 0, ctx->stream>>>(g.ptr.p, g.w.p, n, head.p, mx.p);
    count_launch(ctx);
    ull hm[2];
    SB_CUDA(cudaMemcpyAsync(hm, mx.p, 2 * sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    double wmax;
    memcpy(&wmax, &hm[0], sizeof(double));
    info->max_weight = wmax;
    // the largest sum a vertex can receive in an epoch: as head, per edge one attractive and at most 2 rate + 2 negative
    // contributions; as tail, one per edge; each at most 4 alpha <= 4 learning_rate, rounded
    const double bound = (double)hm[1] * (2.0 * o.rate + 4.0) * (4.0 * o.lr * UM_FIX + 1.0);
    if (!(bound < 4611686018427387904.0))
        return sb_fail(SB_ERR_UNSUPPORTED, "%s: an epoch's position update could pass 2^62 units of 2^-32 (largest degree %llu, learning_rate %g)", fn,
                       (unsigned long long)hm[1], o.lr);
    k_um_prune<<<um_grid(ctx, nnz, 256), 256, 0, ctx->stream>>>(g.w.p, nnz, wmax / (double)n_epochs, keep.p);
    count_launch(ctx);
    SB_TRY(um_select(ctx, head.p, keep.p, ph.p, nnz, num.p));
    SB_TRY(um_select(ctx, g.idx.p, keep.p, pt.p, nnz, num.p));
    SB_TRY(um_select(ctx, g.w.p, keep.p, pw.p, nnz, num.p));
    u64 E = 0;
    SB_CUDA(cudaMemcpyAsync(&E, num.p, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    info->n_edges_used = E;
    head.release();
    keep.release();
    g.idx.release();
    g.w.release();
    DevBuf<double> eps, epn, ens, enn;
    DevBuf<ull> acc;
    SB_TRY(eps.alloc(E));
    SB_TRY(epn.alloc(E));
    SB_TRY(ens.alloc(E));
    SB_TRY(enn.alloc(E));
    SB_TRY(acc.alloc(n * o.nc));
    SB_CUDA(cudaMemsetAsync(acc.p, 0, n * o.nc * sizeof(ull), ctx->stream));
    k_um_schedule<<<um_grid(ctx, E, 256), 256, 0, ctx->stream>>>(pw.p, E, wmax, (double)o.rate, eps.p, epn.p, ens.p, enn.p);
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    pw.release();
    TraceScope te(ctx, "umap: epochs");
    EpochArgs p{ph.p, pt.p, eps.p, epn.p, ens.p, enn.p, Y.p, acc.p, E, n, a, b, b - 1.0, -2.0 * a * b, 2.0 * o.gamma * b, 0.0, 0.0, 0, o.rate > 0};
    const u64 k0 = um_mix64(o.seed);
    for (u32 e = 0; e < n_epochs; e++) {
        p.alpha = o.lr * (1.0 - (double)e / (double)n_epochs);
        p.epoch = (double)e;
        p.key = um_mix64(k0 ^ (u64)e);
        switch (o.nc) {
            case 1: um_launch_epoch<1>(ctx, p); break;
            case 2: um_launch_epoch<2>(ctx, p); break;
            case 3: um_launch_epoch<3>(ctx, p); break;
            case 4: um_launch_epoch<4>(ctx, p); break;
            case 5: um_launch_epoch<5>(ctx, p); break;
            case 6: um_launch_epoch<6>(ctx, p); break;
            case 7: um_launch_epoch<7>(ctx, p); break;
            default: um_launch_epoch<8>(ctx, p); break;
        }
        k_um_apply<<<um_grid(ctx, n * o.nc, 256), 256, 0, ctx->stream>>>(Y.p, acc.p, n * o.nc);
        count_launch(ctx);
        count_launch(ctx);
    }
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

__global__ void k_um_out(const i64 *__restrict__ Y, u64 count, double *__restrict__ out) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (u64)gridDim.x * blockDim.x) out[x] = __dmul_rn((double)Y[x], UM_IFIX);
}
// rows [first, first + count) of Y -> host out
static int um_copy_out(sb_ctx *ctx, const DevBuf<i64> &Y, u64 first, u64 count, u32 nc, double *out) {
    if (!count) return SB_OK;
    DevBuf<double> o;
    SB_TRY(o.alloc(count * nc));
    k_um_out<<<um_grid(ctx, count * nc, 256), 256, 0, ctx->stream>>>(Y.p + first * nc, count * nc, o.p);
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaMemcpyAsync(out, o.p, count * nc * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

static int um_knn_args(const double *X, const uint32_t *nbr, uint64_t n, uint32_t dim, uint32_t k, const char *fn) {
    if (n && (!X || !nbr)) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn);
    if (k == 0) return sb_fail(SB_ERR_INVALID_ARG, "%s: k must be >= 1", fn);
    if (dim == 0) return sb_fail(SB_ERR_INVALID_ARG, "%s: dim must be >= 1", fn);
    if (k > UM_MAX_K) return sb_fail(SB_ERR_UNSUPPORTED, "%s: k must be <= %d", fn, UM_MAX_K);
    if (n >= 0xFFFFFFFFull || n * k >= ((u64)1 << 28)) return sb_fail(SB_ERR_UNSUPPORTED, "%s: n x k must be below 2^28", fn);
    return SB_OK;
}

// the caller's start positions: finite and |value| < 2^30
static int um_user_init(const double *init, u64 rows, u32 nc, const char *fn) {
    if (rows && !init) return sb_fail(SB_ERR_INVALID_ARG, "%s: init must hold n x n_components values", fn);
    for (u64 x = 0; x < rows * nc; x++)
        if (!(std::fabs(init[x]) < UM_INIT_LIMIT)) return sb_fail(SB_ERR_INVALID_ARG, "%s: init values must be finite and below 2^30 in magnitude", fn);
    return SB_OK;
}

// ---------------------------------------------------------------- entry points
extern "C" int sb_umap_graph(sb_ctx *ctx, const double *X, const uint32_t *nbr, uint64_t n, uint32_t dim, uint32_t k, const sb_umap_opts *opts,
                             uint64_t *indptr, uint32_t *indices, double *weights, uint64_t *nnz, double *rho, double *sigma) {
    if (!ctx || !indptr || !nnz || (n && k && (!indices || !weights))) return sb_fail(SB_ERR_INVALID_ARG, "sb_umap_graph: NULL argument");
    UmOpts o;
    SB_TRY(um_opts(opts, o, "sb_umap_graph"));
    SB_TRY(um_knn_args(X, nbr, n, dim, k, "sb_umap_graph"));
    SB_ENTER(ctx);
    DevBuf<double> dX, dr, ds;
    DevBuf<u32> dn;
    SB_TRY(dX.alloc(n * dim));
    SB_TRY(dn.alloc(n * k));
    if (n) {
        SB_CUDA(cudaMemcpyAsync(dX.p, X, n * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(dn.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    }
    UmGraph g;
    SB_TRY(um_graph_build(ctx, dX.p, dn.p, n, dim, k, o.mix, g, dr, ds, "sb_umap_graph"));
    SB_CUDA(cudaMemcpyAsync(indptr, g.ptr.p, (n + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    if (g.nnz) {
        SB_CUDA(cudaMemcpyAsync(indices, g.idx.p, g.nnz * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(weights, g.w.p, g.nnz * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (n && rho) SB_CUDA(cudaMemcpyAsync(rho, dr.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (n && sigma) SB_CUDA(cudaMemcpyAsync(sigma, ds.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    *nnz = g.nnz;
    return SB_OK;
}

// thread per entry: the forward key (i << 32 | j) and the transposed key (j << 32 | i), both with the weight's bits;
// err bit 1 index >= n, 8 a weight outside (0, 1]
__global__ void k_um_pairs(const u64 *__restrict__ ptr, const u32 *__restrict__ idx, const double *__restrict__ w, u64 n, u64 nnz, u64 *__restrict__ fk,
                           u64 *__restrict__ fv, u64 *__restrict__ tk, u64 *__restrict__ tv, int *__restrict__ err) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < nnz; x += (u64)gridDim.x * blockDim.x) {
        u64 lo = 0, hi = n;  // the row: the last i with ptr[i] <= x
        while (hi - lo > 1) {
            const u64 mid = (lo + hi) >> 1;
            if (ptr[mid] <= x) lo = mid;
            else hi = mid;
        }
        const u64 j = idx[x];
        const double v = w[x];
        int e = 0;
        if (j >= n) e |= 1;
        if (!(v > 0.0 && v <= 1.0)) e |= 8;
        if (e) atomicOr(err, e);
        fk[x] = (lo << 32) | j;
        tk[x] = (j << 32) | lo;
        fv[x] = tv[x] = (u64)__double_as_longlong(v);
    }
}
// thread per entry of the row-sorted copy: bit 2 asymmetric (pair or weight), 4 duplicate entry
__global__ void k_um_check(const u64 *__restrict__ fk, const u64 *__restrict__ fv, const u64 *__restrict__ tk, const u64 *__restrict__ tv, u64 nnz,
                           int *__restrict__ err) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < nnz; x += (u64)gridDim.x * blockDim.x) {
        int e = 0;
        if (fk[x] != tk[x] || fv[x] != tv[x]) e |= 2;
        if (x && fk[x] == fk[x - 1]) e |= 4;
        if (e) atomicOr(err, e);
    }
}

int um_csr_host_check(u64 n, const u64 *indptr, const u32 *indices, const double *weights, const char *fn) {
    if (n >= 0xFFFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "%s: more than 2^32 - 2 vertices", fn);
    if (indptr[0] != 0) return sb_fail(SB_ERR_INVALID_ARG, "%s: indptr must start at 0", fn);
    for (u64 i = 0; i < n; i++)
        if (indptr[i + 1] < indptr[i]) return sb_fail(SB_ERR_INVALID_ARG, "%s: indptr decreases at row %llu", fn, (unsigned long long)i);
    if (indptr[n] && (!indices || !weights)) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn);
    return SB_OK;
}

int um_csr_upload(sb_ctx *ctx, u64 n, const u64 *indptr, const u32 *indices, const double *weights, UmGraph &g, const char *fn,
                  const char *trace) {
    const u64 nnz = indptr[n];
    g.n = n;
    g.nnz = nnz;
    SB_TRY(g.ptr.alloc(n + 1));
    SB_CUDA(cudaMemcpyAsync(g.ptr.p, indptr, (n + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    if (!nnz) return SB_OK;
    // validation: the row-sorted pairs must equal the sorted transposed pairs, weights included, with no repeated pair
    TraceScope tr(ctx, trace);
    DevBuf<u32> di;
    DevBuf<double> dw;
    DevBuf<u64> fk, fv, tk, tv;
    DevBuf<int> err;
    SB_TRY(di.alloc(nnz));
    SB_TRY(dw.alloc(nnz));
    SB_TRY(fk.alloc(nnz));
    SB_TRY(fv.alloc(nnz));
    SB_TRY(tk.alloc(nnz));
    SB_TRY(tv.alloc(nnz));
    SB_TRY(err.alloc(1));
    SB_CUDA(cudaMemcpyAsync(di.p, indices, nnz * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(dw.p, weights, nnz * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), ctx->stream));
    k_um_pairs<<<um_grid(ctx, nnz, 256), 256, 0, ctx->stream>>>(g.ptr.p, di.p, dw.p, n, nnz, fk.p, fv.p, tk.p, tv.p, err.p);
    count_launch(ctx);
    SB_TRY(sort_pairs(ctx, fk, fv, nnz));
    SB_TRY(sort_pairs(ctx, tk, tv, nnz));
    k_um_check<<<um_grid(ctx, nnz, 256), 256, 0, ctx->stream>>>(fk.p, fv.p, tk.p, tv.p, nnz, err.p);
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    int herr = 0;
    SB_CUDA(cudaMemcpyAsync(&herr, err.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (herr & 1) return sb_fail(SB_ERR_INVALID_ARG, "%s: a column index >= n", fn);
    if (herr & 8) return sb_fail(SB_ERR_INVALID_ARG, "%s: a weight outside (0, 1]", fn);
    if (herr & 4) return sb_fail(SB_ERR_INVALID_ARG, "%s: a duplicate entry", fn);
    if (herr & 2) return sb_fail(SB_ERR_INVALID_ARG, "%s: the CSR is not symmetric (pairs or weights)", fn);
    // the graph: columns ascending
    SB_TRY(um_rows_from_keys(ctx, fk.p, g));
    SB_TRY(g.w.alloc(nnz));
    SB_CUDA(cudaMemcpyAsync(g.w.p, fv.p, nnz * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    return SB_OK;
}

extern "C" int sb_umap_layout(sb_ctx *ctx, uint64_t n, const uint64_t *indptr, const uint32_t *indices, const double *weights, const double *init,
                              const sb_umap_opts *opts, double *out, sb_umap_info *info) {
    if (!ctx || !indptr || !info || (n && !out)) return sb_fail(SB_ERR_INVALID_ARG, "sb_umap_layout: NULL argument");
    UmOpts o;
    SB_TRY(um_opts(opts, o, "sb_umap_layout"));
    SB_TRY(um_csr_host_check(n, indptr, indices, weights, "sb_umap_layout"));
    if (o.init != SB_UMAP_INIT_RANDOM) SB_TRY(um_user_init(init, n, o.nc, "sb_umap_layout"));
    SB_ENTER(ctx);
    UmGraph g;
    SB_TRY(um_csr_upload(ctx, n, indptr, indices, weights, g, "sb_umap_layout", "umap: csr validation"));
    DevBuf<double> dA;
    SB_TRY(dA.alloc(n * o.nc));
    if (n && o.init != SB_UMAP_INIT_RANDOM) SB_CUDA(cudaMemcpyAsync(dA.p, init, n * o.nc * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    DevBuf<i64> Y;
    SB_TRY(um_init(ctx, dA.p, n, o.nc, o, Y));
    SB_TRY(um_layout(ctx, g, Y, o, info, "sb_umap_layout"));
    return um_copy_out(ctx, Y, 0, n, o.nc, out);
}

int um_gather_rows(sb_ctx *ctx, const void *mine_h, u64 n_local, u64 width_words, const std::vector<u64> &counts, u64 maxr, u32 *dst) {
    const u64 slab = maxr * width_words;
    DevBuf<u32> mine, all;
    SB_TRY(mine.alloc(slab));
    SB_TRY(all.alloc(slab * ctx->nranks));
    SB_CUDA(cudaMemsetAsync(mine.p, 0, std::max<u64>(1, slab) * sizeof(u32), ctx->stream));
    if (n_local) SB_CUDA(cudaMemcpyAsync(mine.p, mine_h, n_local * width_words * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    if (slab) {
        ProfScope ps(ctx, PH_COMM);
        SB_NCCL(ncclAllGather(mine.p, all.p, slab, ncclUint32, ctx->comm, ctx->stream));
        count_launch(ctx, false);
    }
    u64 at = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        if (counts[r])
            SB_CUDA(cudaMemcpyAsync(dst + at * width_words, all.p + (u64)r * slab, counts[r] * width_words * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));
        at += counts[r];
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

extern "C" int sb_umap(sb_ctx *ctx, const double *X, const uint32_t *nbr, uint64_t n_local, uint32_t dim, uint32_t k, const sb_umap_opts *opts,
                       const double *init, double *out, sb_umap_info *info) {
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "sb_umap: NULL argument");
    UmOpts o;
    int rc = (!info || (n_local && !out)) ? sb_fail(SB_ERR_INVALID_ARG, "sb_umap: NULL argument") : SB_OK;
    if (rc == SB_OK) rc = um_opts(opts, o, "sb_umap");
    if (rc == SB_OK) rc = um_knn_args(X, nbr, n_local, dim, k, "sb_umap");
    if (rc == SB_OK && o.nc > dim && o.init == SB_UMAP_INIT_PCA) rc = sb_fail(SB_ERR_INVALID_ARG, "sb_umap: pca init needs n_components <= dim");
    if (rc == SB_OK && o.init == SB_UMAP_INIT_USER) rc = um_user_init(init, n_local, o.nc, "sb_umap");
    SB_ENTER(ctx);
    SB_TRY(agree_status(ctx, rc, "sb_umap"));
    std::vector<u64> counts, shape;
    SB_TRY(comm_allgather_u64_host(ctx, n_local, counts));
    SB_TRY(comm_allgather_u64_host(ctx, ((u64)k << 32) | dim, shape));
    u64 n = 0, maxr = 0, off = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        if (shape[r] != (((u64)k << 32) | dim)) return sb_fail(SB_ERR_INVALID_ARG, "sb_umap: k or dim differs between ranks (rank %d)", r);
        if (r < ctx->rank) off += counts[r];
        n += counts[r];
        maxr = std::max(maxr, counts[r]);
    }
    if (n >= 0xFFFFFFFFull || n * k >= ((u64)1 << 28)) return sb_fail(SB_ERR_UNSUPPORTED, "sb_umap: n x k must be below 2^28 over all ranks");
    DevBuf<double> dX, dU;
    DevBuf<u32> dn;
    SB_TRY(dX.alloc(n * dim));
    SB_TRY(dn.alloc(n * k));
    SB_TRY(dU.alloc(o.init == SB_UMAP_INIT_USER ? n * o.nc : 0));
    if (ctx->nranks == 1) {
        if (n) {
            SB_CUDA(cudaMemcpyAsync(dX.p, X, n * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            SB_CUDA(cudaMemcpyAsync(dn.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
            if (o.init == SB_UMAP_INIT_USER) SB_CUDA(cudaMemcpyAsync(dU.p, init, n * o.nc * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        }
    } else {
        TraceScope tr(ctx, "umap: row all-gather");
        SB_TRY(um_gather_rows(ctx, X, n_local, 2 * (u64)dim, counts, maxr, (u32 *)dX.p));
        SB_TRY(um_gather_rows(ctx, nbr, n_local, k, counts, maxr, dn.p));
        if (o.init == SB_UMAP_INIT_USER) SB_TRY(um_gather_rows(ctx, init, n_local, 2 * (u64)o.nc, counts, maxr, (u32 *)dU.p));
    }
    UmGraph g;
    DevBuf<double> dr, ds;
    SB_TRY(um_graph_build(ctx, dX.p, dn.p, n, dim, k, o.mix, g, dr, ds, "sb_umap"));
    dn.release();
    dr.release();
    ds.release();
    DevBuf<i64> Y;
    if (o.init == SB_UMAP_INIT_USER) SB_TRY(um_init(ctx, dU.p, n, o.nc, o, Y));
    else SB_TRY(um_init(ctx, dX.p, n, dim, o, Y));
    dX.release();
    dU.release();
    SB_TRY(um_layout(ctx, g, Y, o, info, "sb_umap"));
    return um_copy_out(ctx, Y, off, n_local, o.nc, out);
}

// ---------------------------------------------------------------- transform: new points into a fixed reference embedding
// umap-learn's transform with move_other = False: only the query point (the head) moves, and a head's entries are its own, so one
// thread per query row runs every epoch with its entries in slot order and adds every contribution at once.  That is umap-learn's
// loop (epochs outside, entries inside) bit for bit, in one launch, without atomics.

// thread per row of the n x k weights: the start (umap-learn's init_graph_transform, slots in order) into Y; the largest weight
// (positive doubles order as their bits) and the entries with w > 0 into mx[0], mx[1]; err bits 32 a weight outside [0, 1], 64 a
// row whose weights are all 0
__global__ void k_ut_start(const u32 *__restrict__ nbr, const double *__restrict__ w, u64 n, u32 k, u32 nc, const i64 *__restrict__ E,
                           i64 *__restrict__ Y, ull *__restrict__ mx, int *__restrict__ err) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const double *wi = w + i * k;
        const u32 *ri = nbr + i * k;
        double rs = 0.0;
        ull m = 0, pos = 0;
        u32 one = k;
        int e = 0;
        for (u32 t = 0; t < k; t++) {
            const double v = wi[t];
            if (!(v >= 0.0 && v <= 1.0)) e |= 32;
            rs = __dadd_rn(rs, v);
            if (v > 0.0) pos++;
            if (v == 1.0 && one == k) one = t;
            const ull b = (ull)__double_as_longlong(v);
            m = v > 0.0 && b > m ? b : m;
        }
        if (!e && !(rs > 0.0)) e |= 64;
        if (e) {
            atomicOr(err, e);
            continue;
        }
        for (u32 c = 0; c < nc; c++) {
            if (one < k) {
                Y[i * nc + c] = E[(u64)ri[one] * nc + c];
                continue;
            }
            double acc = 0.0;
            for (u32 t = 0; t < k; t++)
                acc = __dadd_rn(acc, __dmul_rn(__ddiv_rn(wi[t], rs), __dmul_rn((double)E[(u64)ri[t] * nc + c], UM_IFIX)));
            Y[i * nc + c] = __double2ll_rn(__dmul_rn(acc, UM_FIX));
        }
        if (m) atomicMax(&mx[0], m);
        atomicAdd(&mx[1], pos);
    }
}

struct UtArgs {
    const u32 *nbr;      // [n x k] reference indices
    const double *w;     // [n x k]
    const i64 *E;        // [n_ref x NC] the reference, units of 2^-32 (never written)
    i64 *Y;              // [n x NC] the start in, the result out
    double *ens, *enn;   // [k x n] next epoch of each entry and of its negative samples
    ull *used;           // entries left after pruning
    u64 n, n_ref, row0;  // row0: the global index of local row 0
    u32 k, n_epochs;
    double wmax, thr, rate, a, b, bm1, m2ab, two_gb, alpha0;
    u64 key0;            // mix64(seed)
    int negatives;
};

// thread per query row, every epoch
template <int NC>
__global__ void __launch_bounds__(128) k_ut_layout(UtArgs p) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += (u64)gridDim.x * blockDim.x) {
        i64 y[NC];
#pragma unroll
        for (int c = 0; c < NC; c++) y[c] = p.Y[i * NC + c];
        const double *wi = p.w + i * p.k;
        const u32 *ri = p.nbr + i * p.k;
        ull used = 0;
        for (u32 t = 0; t < p.k; t++) {  // prune and schedule: eps = w_max / w, epn = eps / rate; next = eps, next_neg = epn
            const double v = wi[t];
            const bool keep = v >= p.thr;
            const double eps = keep ? __ddiv_rn(p.wmax, v) : INFINITY;
            p.ens[(u64)t * p.n + i] = eps;
            p.enn[(u64)t * p.n + i] = p.negatives ? __ddiv_rn(eps, p.rate) : INFINITY;
            used += keep;
        }
        if (used) atomicAdd(p.used, used);
        for (u32 ep = 0; ep < p.n_epochs; ep++) {
            const double epoch = (double)ep;
            const double alpha = __dmul_rn(p.alpha0, __dsub_rn(1.0, __ddiv_rn(epoch, (double)p.n_epochs)));
            const u64 key = um_mix64(p.key0 ^ (u64)ep);
            for (u32 t = 0; t < p.k; t++) {
                double *ens = p.ens + (u64)t * p.n + i;
                const double ns = *ens;
                if (ns > epoch) continue;
                const u64 j = ri[t];
                double yi[NC], yk[NC];
                double d2 = 0.0;
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    yi[c] = __dmul_rn((double)y[c], UM_IFIX);
                    yk[c] = __dmul_rn((double)p.E[j * NC + c], UM_IFIX);
                    const double df = __dsub_rn(yi[c], yk[c]);
                    d2 = __dadd_rn(d2, __dmul_rn(df, df));
                }
                const double gc = d2 > 0.0 ? __ddiv_rn(__dmul_rn(p.m2ab, pow(d2, p.bm1)), __dadd_rn(__dmul_rn(p.a, pow(d2, p.b)), 1.0)) : 0.0;
#pragma unroll
                for (int c = 0; c < NC; c++) y[c] += um_fix(um_clip(__dmul_rn(gc, __dsub_rn(yi[c], yk[c]))), alpha);
                const double eps = __ddiv_rn(p.wmax, wi[t]);
                *ens = __dadd_rn(ns, eps);
                if (!p.negatives) continue;
                double *enn = p.enn + (u64)t * p.n + i;
                const double epn = __ddiv_rn(eps, p.rate), nn_f = *enn;
                i64 nn = (i64)__ddiv_rn(__dsub_rn(epoch, nn_f), epn);
                if (nn < 0) nn = 0;
                const u64 k2 = um_mix64(key ^ ((p.row0 + i) * p.k + t));
                for (i64 s = 0; s < nn; s++) {
                    const u64 v = um_mix64(k2 ^ (u64)s) % p.n_ref;
                    double dd = 0.0;
#pragma unroll
                    for (int c = 0; c < NC; c++) {
                        yi[c] = __dmul_rn((double)y[c], UM_IFIX);
                        yk[c] = __dmul_rn((double)p.E[v * NC + c], UM_IFIX);
                        const double df = __dsub_rn(yi[c], yk[c]);
                        dd = __dadd_rn(dd, __dmul_rn(df, df));
                    }
                    if (dd > 0.0) {
                        const double g = __ddiv_rn(p.two_gb, __dmul_rn(__dadd_rn(0.001, dd), __dadd_rn(__dmul_rn(p.a, pow(dd, p.b)), 1.0)));
#pragma unroll
                        for (int c = 0; c < NC; c++) y[c] += um_fix(um_clip(__dmul_rn(g, __dsub_rn(yi[c], yk[c]))), alpha);
                    } else {
                        const i64 f = um_fix(4.0, alpha);
#pragma unroll
                        for (int c = 0; c < NC; c++) y[c] += f;
                    }
                }
                *enn = __dadd_rn(nn_f, __dmul_rn((double)nn, epn));
            }
        }
#pragma unroll
        for (int c = 0; c < NC; c++) p.Y[i * NC + c] = y[c];
    }
}

template <int NC>
static void ut_launch_layout(sb_ctx *ctx, const UtArgs &a) {
    k_ut_layout<NC><<<um_grid(ctx, a.n, 128), 128, 0, ctx->stream>>>(a);
}

// the entry points' host checks (k, n_ref, sizes; opts with init and set_op_mix_ratio ignored); NULL pointers are the caller's
static int ut_args(const sb_umap_opts *opts, u64 n_ref, u64 n, u32 k, UmOpts &o, const char *fn) {
    sb_umap_opts c = opts ? *opts : sb_umap_opts{2, 0, 0.1, 1.0, 0.0, 0.0, 1.0, 1.0, 1.0, 5, SB_UMAP_INIT_PCA, 0};
    c.init = SB_UMAP_INIT_PCA;
    c.set_op_mix_ratio = 1.0;
    SB_TRY(um_opts(&c, o, fn));
    if (k < 2) return sb_fail(SB_ERR_INVALID_ARG, "%s: k must be >= 2", fn);
    if (k > UM_MAX_K) return sb_fail(SB_ERR_UNSUPPORTED, "%s: k must be <= %d", fn, UM_MAX_K);
    if (n_ref >= 0xFFFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "%s: n_ref must be below 2^32 - 1", fn);
    if (k > n_ref) return sb_fail(SB_ERR_INVALID_ARG, "%s: k must be <= n_ref", fn);
    if (n * k >= ((u64)1 << 28)) return sb_fail(SB_ERR_UNSUPPORTED, "%s: n x k must be below 2^28", fn);
    return SB_OK;
}

// the reference embedding [n_ref x nc]: finite and |e| < 2^30
static int ut_ref_embedding(const double *e, u64 n_ref, u32 nc, const char *fn) {
    if (!e) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn);
    for (u64 x = 0; x < n_ref * nc; x++)
        if (!(std::fabs(e[x]) < UM_INIT_LIMIT)) return sb_fail(SB_ERR_INVALID_ARG, "%s: ref_embedding values must be finite and below 2^30 in magnitude", fn);
    return SB_OK;
}

// the device error bits of k_um_dist / k_ut_start -> a status (agreed over the ranks by the caller)
static int ut_err(int e, const char *fn) {
    if (!e) return SB_OK;
    return sb_fail(SB_ERR_INVALID_ARG, "%s: invalid neighbour lists or weights:%s%s%s%s%s", fn, e & 1 ? " an index >= n_ref" : "",
                   e & 4 ? " a duplicate in a row" : "", e & 24 ? " padding (rows must be full)" : "", e & 32 ? " a weight outside [0, 1]" : "",
                   e & 64 ? " a row whose weights are all 0" : "");
}

// every rank's row count -> the global query count and this rank's first row; k must agree
static int ut_rows(sb_ctx *ctx, u64 n, u32 k, u64 &n_global, u64 &row0, const char *fn) {
    std::vector<u64> counts, ks;
    SB_TRY(comm_allgather_u64_host(ctx, n, counts));
    SB_TRY(comm_allgather_u64_host(ctx, k, ks));
    n_global = row0 = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        if (ks[r] != k) return sb_fail(SB_ERR_INVALID_ARG, "%s: k differs between ranks (rank %d)", fn, r);
        if (r < ctx->rank) row0 += counts[r];
        n_global += counts[r];
    }
    return SB_OK;
}

// the query rows' graph: X [n x dim] against the reference R [n_ref x dim], nbr [n x k] on the device -> w [n x k], sigma [n]
static int ut_graph(sb_ctx *ctx, const double *R, u64 n_ref, const double *X, const u32 *nbr, u64 n, u32 dim, u32 k, DevBuf<double> &w,
                    DevBuf<double> &sigma, const char *fn) {
    TraceScope tr(ctx, "umap transform: graph");
    const u64 nk = n * k;
    DevBuf<double> d, rho, rs;
    DevBuf<int> flags;  // [0] error bits, [1] unused (every rho is 0)
    DevBuf<ull> cnt;
    SB_TRY(d.alloc(nk));
    SB_TRY(w.alloc(nk));
    SB_TRY(rho.alloc(n));
    SB_TRY(rs.alloc(n));
    SB_TRY(sigma.alloc(n));
    SB_TRY(flags.alloc(2));
    SB_TRY(cnt.alloc(1));
    SB_CUDA(cudaMemsetAsync(flags.p, 0, 2 * sizeof(int), ctx->stream));
    SB_CUDA(cudaMemsetAsync(cnt.p, 0, sizeof(ull), ctx->stream));
    if (n) {
        k_um_dist<<<um_grid(ctx, nk, 256), 256, 0, ctx->stream>>>(X, R, n_ref, nbr, n, dim, k, 1, d.p, flags.p);
        k_um_smooth<<<um_grid(ctx, n, 128), 128, 0, ctx->stream>>>(d.p, nbr, n, k, std::log2((double)k), 1, rho.p, sigma.p, rs.p, flags.p + 1, cnt.p);
        count_launch(ctx);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
    }
    int hf[2];
    SB_CUDA(cudaMemcpyAsync(hf, flags.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_TRY(agree_status(ctx, ut_err(hf[0], fn), fn));
    // the global floor: the row sums of all ranks in global row order, summed left to right; sum m by the integer all-reduce
    std::vector<double> mine(n), all;
    if (n) SB_CUDA(cudaMemcpyAsync(mine.data(), rs.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_TRY(gather_cells(ctx, mine, all));
    SB_TRY(comm_allreduce_u64(ctx, (u64 *)cnt.p, 1));
    ull hc = 0;
    SB_CUDA(cudaMemcpyAsync(&hc, cnt.p, sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    double tot = 0.0;
    for (double v : all) tot += v;
    if (n) {
        k_um_global_floor<<<um_grid(ctx, n, 256), 256, 0, ctx->stream>>>(rho.p, sigma.p, n, 1e-3 * (tot / (double)hc));
        k_um_member<<<um_grid(ctx, nk, 256), 256, 0, ctx->stream>>>(d.p, nbr, n, k, rho.p, sigma.p, w.p, nullptr, nullptr);
        count_launch(ctx);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// the start and the epochs from the reference embedding (host, checked) and the query rows' nbr and w on the device -> host out
static int ut_layout(sb_ctx *ctx, const double *ref_embedding, u64 n_ref, const u32 *nbr, const double *w, u64 n, u32 k, const UmOpts &o,
                     double *out, sb_umap_info *info, const char *fn) {
    TraceScope tr(ctx, "umap transform: start");
    const u32 nc = o.nc;
    DevBuf<double> dA;
    DevBuf<i64> E, Y;
    DevBuf<ull> mx;
    DevBuf<int> err;
    SB_TRY(dA.alloc(n_ref * nc));
    SB_TRY(E.alloc(n_ref * nc));
    SB_TRY(Y.alloc(n * nc));
    SB_TRY(mx.alloc(3));
    SB_TRY(err.alloc(1));
    SB_CUDA(cudaMemsetAsync(mx.p, 0, 3 * sizeof(ull), ctx->stream));
    SB_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), ctx->stream));
    SB_CUDA(cudaMemcpyAsync(dA.p, ref_embedding, n_ref * nc * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    k_um_init<<<um_grid(ctx, n_ref * nc, 256), 256, 0, ctx->stream>>>(dA.p, n_ref, nc, nc, 2, nullptr, nullptr, 0, E.p);
    count_launch(ctx);
    if (n) {
        k_ut_start<<<um_grid(ctx, n, 128), 128, 0, ctx->stream>>>(nbr, w, n, k, nc, E.p, Y.p, mx.p, err.p);
        count_launch(ctx);
    }
    SB_CUDA(cudaGetLastError());
    ull hm[2];
    int herr = 0;
    SB_CUDA(cudaMemcpyAsync(hm, mx.p, 2 * sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(&herr, err.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    dA.release();
    SB_TRY(agree_status(ctx, ut_err(herr, fn), fn));
    // the global quantities: the query count and this rank's first row, w_max (max over the ranks) and the entries with w > 0
    u64 n_global = 0, row0 = 0;
    SB_TRY(ut_rows(ctx, n, k, n_global, row0, fn));
    std::vector<u64> wm, pos;
    SB_TRY(comm_allgather_u64_host(ctx, hm[0], wm));
    SB_TRY(comm_allgather_u64_host(ctx, hm[1], pos));
    u64 wbits = 0, n_pos = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        wbits = std::max(wbits, wm[r]);
        n_pos += pos[r];
    }
    double wmax;
    memcpy(&wmax, &wbits, sizeof(double));
    double a = o.a, b = o.b;
    if (!(a > 0.0 && b > 0.0)) um_fit_ab(o.spread, o.min_dist, a, b);
    const u32 n_epochs = o.n_epochs ? o.n_epochs / 3 : (n_global <= 10000 ? 100 : 30);
    info->a = a;
    info->b = b;
    info->max_weight = wmax;
    info->n_edges = n_pos;
    info->n_edges_used = 0;
    info->n_epochs = n_epochs;
    if (n_epochs && n_global) {
        // the most a point can move over all epochs: per epoch and entry one attractive and at most 2 rate + 2 negative
        // contributions, each at most 4 alpha <= learning_rate, rounded
        const double bound = (double)n_epochs * k * (2.0 * o.rate + 4.0) * (o.lr * UM_FIX + 1.0);
        if (!(bound < 4611686018427387904.0))
            return sb_fail(SB_ERR_UNSUPPORTED, "%s: the epochs could move a point by 2^62 units of 2^-32 (k %u, %u epochs, learning_rate %g)", fn, k,
                           n_epochs, o.lr);
        TraceScope te(ctx, "umap transform: epochs");
        DevBuf<double> ens, enn;
        SB_TRY(ens.alloc(n * k));
        SB_TRY(enn.alloc(n * k));
        UtArgs p{nbr, w, E.p, Y.p, ens.p, enn.p, mx.p + 2, n, n_ref, row0, k, n_epochs, wmax, wmax / (double)n_epochs, (double)o.rate, a, b,
                 b - 1.0, -2.0 * a * b, 2.0 * o.gamma * b, o.lr / 4.0, um_mix64(o.seed), o.rate > 0};
        if (n) {
            switch (nc) {
                case 1: ut_launch_layout<1>(ctx, p); break;
                case 2: ut_launch_layout<2>(ctx, p); break;
                case 3: ut_launch_layout<3>(ctx, p); break;
                case 4: ut_launch_layout<4>(ctx, p); break;
                case 5: ut_launch_layout<5>(ctx, p); break;
                case 6: ut_launch_layout<6>(ctx, p); break;
                case 7: ut_launch_layout<7>(ctx, p); break;
                default: ut_launch_layout<8>(ctx, p); break;
            }
            count_launch(ctx);
            SB_CUDA(cudaGetLastError());
        }
        ull used = 0;
        SB_CUDA(cudaMemcpyAsync(&used, mx.p + 2, sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        std::vector<u64> us;
        SB_TRY(comm_allgather_u64_host(ctx, used, us));
        for (u64 v : us) info->n_edges_used += v;
    }
    return um_copy_out(ctx, Y, 0, n, nc, out);
}

extern "C" int sb_umap_transform_graph(sb_ctx *ctx, const double *ref_scores, uint64_t n_ref, const double *scores, const uint32_t *nbr, uint64_t n,
                                       uint32_t dim, uint32_t k, const sb_umap_opts *opts, double *weights, double *sigma) {
    const char *fn = "sb_umap_transform_graph";
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn);
    UmOpts o;
    int rc = (!ref_scores || (n && (!scores || !nbr || !weights))) ? sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn) : SB_OK;
    if (rc == SB_OK && dim == 0) rc = sb_fail(SB_ERR_INVALID_ARG, "%s: dim must be >= 1", fn);
    if (rc == SB_OK) rc = ut_args(opts, n_ref, n, k, o, fn);
    SB_ENTER(ctx);
    SB_TRY(agree_status(ctx, rc, fn));
    DevBuf<double> dR, dX, w, s;
    DevBuf<u32> dn;
    SB_TRY(dR.alloc(n_ref * dim));
    SB_TRY(dX.alloc(n * dim));
    SB_TRY(dn.alloc(n * k));
    SB_CUDA(cudaMemcpyAsync(dR.p, ref_scores, n_ref * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    if (n) {
        SB_CUDA(cudaMemcpyAsync(dX.p, scores, n * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(dn.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    }
    SB_TRY(ut_graph(ctx, dR.p, n_ref, dX.p, dn.p, n, dim, k, w, s, fn));
    if (n) {
        SB_CUDA(cudaMemcpyAsync(weights, w.p, n * k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        if (sigma) SB_CUDA(cudaMemcpyAsync(sigma, s.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

extern "C" int sb_umap_transform_layout(sb_ctx *ctx, const double *ref_embedding, uint64_t n_ref, const uint32_t *nbr, const double *weights, uint64_t n,
                                        uint32_t k, const sb_umap_opts *opts, double *out, sb_umap_info *info) {
    const char *fn = "sb_umap_transform_layout";
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn);
    UmOpts o;
    int rc = (!info || (n && (!nbr || !weights || !out))) ? sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn) : SB_OK;
    if (rc == SB_OK) rc = ut_args(opts, n_ref, n, k, o, fn);
    if (rc == SB_OK) rc = ut_ref_embedding(ref_embedding, n_ref, o.nc, fn);
    SB_ENTER(ctx);
    SB_TRY(agree_status(ctx, rc, fn));
    DevBuf<double> dw, d;
    DevBuf<u32> dn;
    DevBuf<int> err;
    SB_TRY(dw.alloc(n * k));
    SB_TRY(dn.alloc(n * k));
    SB_TRY(d.alloc(n * k));
    SB_TRY(err.alloc(1));
    SB_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), ctx->stream));
    if (n) {
        SB_CUDA(cudaMemcpyAsync(dn.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(dw.p, weights, n * k * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        // the neighbour lists' checks of the graph step (dim 0: no distance is computed)
        k_um_dist<<<um_grid(ctx, n * k, 256), 256, 0, ctx->stream>>>(nullptr, nullptr, n_ref, dn.p, n, 0, k, 1, d.p, err.p);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
    }
    int herr = 0;
    SB_CUDA(cudaMemcpyAsync(&herr, err.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    d.release();
    SB_TRY(agree_status(ctx, ut_err(herr, fn), fn));
    return ut_layout(ctx, ref_embedding, n_ref, dn.p, dw.p, n, k, o, out, info, fn);
}

extern "C" int sb_umap_transform(sb_ctx *ctx, const double *ref_scores, const double *ref_embedding, uint64_t n_ref, const double *scores,
                                 const uint32_t *nbr, uint64_t n_local, uint32_t dim, uint32_t k, const sb_umap_opts *opts, double *out,
                                 sb_umap_info *info) {
    const char *fn = "sb_umap_transform";
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn);
    UmOpts o;
    int rc = (!ref_scores || !info || (n_local && (!scores || !nbr || !out))) ? sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn) : SB_OK;
    if (rc == SB_OK && dim == 0) rc = sb_fail(SB_ERR_INVALID_ARG, "%s: dim must be >= 1", fn);
    if (rc == SB_OK) rc = ut_args(opts, n_ref, n_local, k, o, fn);
    if (rc == SB_OK) rc = ut_ref_embedding(ref_embedding, n_ref, o.nc, fn);
    SB_ENTER(ctx);
    SB_TRY(agree_status(ctx, rc, fn));
    const u64 n = n_local;
    DevBuf<double> dR, dX, w, s;
    DevBuf<u32> dn;
    SB_TRY(dR.alloc(n_ref * dim));
    SB_TRY(dX.alloc(n * dim));
    SB_TRY(dn.alloc(n * k));
    SB_CUDA(cudaMemcpyAsync(dR.p, ref_scores, n_ref * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    if (n) {
        SB_CUDA(cudaMemcpyAsync(dX.p, scores, n * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(dn.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    }
    SB_TRY(ut_graph(ctx, dR.p, n_ref, dX.p, dn.p, n, dim, k, w, s, fn));
    dR.release();
    dX.release();
    s.release();
    return ut_layout(ctx, ref_embedding, n_ref, dn.p, w.p, n, k, o, out, info, fn);
}
