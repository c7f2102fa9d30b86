// tsne.cu -- the t-SNE embedding of the kNN lists (the reference workspace's `bhtsne` crate, van der Maaten's Barnes-Hut t-SNE):
// perplexity-calibrated affinities and a deterministic Barnes-Hut layout.  The rules are stated beside the entry points in
// include/scanb200.h and restated by oracle/tsne.py.  Compiled with -fmad=false: every + - x / sqrt below is one correctly rounded
// operation, so the layout equals the oracle bit for bit from a given P and start.
//
//   affinities  the scores zero-meaned per column and divided by their largest |x| (k_ts_part / k_ts_fin / k_ts_scale);
//               k_um_dist on them, D = d d; k_ts_beta: a thread per row runs bhtsne's beta search; the symmetric P is the pair-key
//               sort of UMAP's fuzzy union (forward and transposed keys, k_ts_join adds P_ij + P_ji, a flagged select), divided by
//               its total summed in chunks of TS_CHUNK entries.
//   layout      per iteration: the root box (k_ts_part / k_ts_fin over Y), 64-bit Morton codes (k_ts_codes) sorted with the cell
//               index as value, runs of equal codes as leaves (k_ts_runs + a scan + k_ts_leaves), Karras' radix tree over the
//               distinct codes (k_ts_karras), leaf sums in sorted order and internal sums left + right by the second thread up
//               (k_ts_sums), then a thread per point in Morton order: attractive forces over its CSR row and the Barnes-Hut walk
//               (k_ts_forces); sum_Q (k_ts_part / k_ts_fin over the per-point sums), the gains update (k_ts_update), zero mean
//               (k_ts_center).  No host round trip inside the loop.
//
// Every sum whose order could vary with the launch is taken in chunks: chunk c holds elements [c TS_CHUNK, (c + 1) TS_CHUNK), each
// chunk is summed left to right from its first element, and the chunk sums left to right; so the order depends on the count alone.
#include <cfloat>
#include <cmath>

#include <cub/cub.cuh>

#include "common.cuh"

#define TS_PAD 0xFFFFFFFFu
#define TS_MAX_K 128
#define TS_CHUNK 1024
#define TS_TAG (1ull << 63)
#define TS_LEAF 0x80000000u
#define TS_STACK 72  // a walk holds at most one pending sibling per level; prefixes grow by >= 1 bit per level (<= 64 + a leaf)

typedef unsigned long long ull;

static int ts_grid(sb_ctx *ctx, u64 items, int per_block) {
    return (int)std::max<u64>(1, std::min<u64>((items + per_block - 1) / per_block, (u64)ctx->sm_count * 32));
}

// ---------------------------------------------------------------- ordered sums
// thread per (chunk, column) of A [n x ld], columns < ncol: the chunk's sum left to right from its first element (of (a - c[col])^2
// when c is given), its min and max
__global__ void k_ts_part(const double *__restrict__ A, u32 ld, u32 ncol, u64 n, const double *__restrict__ c, double *__restrict__ sum,
                          double *__restrict__ mn, double *__restrict__ mx) {
    const u64 nch = (n + TS_CHUNK - 1) / TS_CHUNK;
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nch * ncol; t += (u64)gridDim.x * blockDim.x) {
        const u64 ch = t / ncol, col = t - ch * ncol, lo = ch * TS_CHUNK, hi = std::min<u64>(n, lo + TS_CHUNK);
        const double cc = c ? c[col] : 0.0;
        double s = 0.0, l = INFINITY, h = -INFINITY;
        for (u64 i = lo; i < hi; i++) {
            double v = A[i * ld + col];
            l = fmin(l, v);
            h = fmax(h, v);
            if (c) {
                v = v - cc;
                v = v * v;
            }
            s = i == lo ? v : s + v;
        }
        sum[t] = s;
        mn[t] = l;
        mx[t] = h;
    }
}
// thread per column: the chunk sums left to right (divided by n when mean), the min and max -> out[3 col + 0, 1, 2]
__global__ void k_ts_fin(const double *__restrict__ sum, const double *__restrict__ mn, const double *__restrict__ mx, u64 nch, u32 ncol, u64 n,
                         int mean, double *__restrict__ out) {
    const u32 col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= ncol) return;
    double s = 0.0, l = INFINITY, h = -INFINITY;
    for (u64 ch = 0; ch < nch; ch++) {
        const u64 t = ch * ncol + col;
        s = ch == 0 ? sum[t] : s + sum[t];
        l = fmin(l, mn[t]);
        h = fmax(h, mx[t]);
    }
    out[3 * col] = mean ? s / (double)n : s;
    out[3 * col + 1] = l;
    out[3 * col + 2] = h;
}

// Workspace of the ordered sums over up to n rows x ncol columns.
struct TsSum {
    DevBuf<double> sum, mn, mx;
    u64 cap = 0;
    int init(u64 n, u32 ncol) {
        cap = std::max<u64>(1, (n + TS_CHUNK - 1) / TS_CHUNK) * ncol;
        SB_TRY(sum.alloc(cap));
        SB_TRY(mn.alloc(cap));
        SB_TRY(mx.alloc(cap));
        return SB_OK;
    }
    // out[3 col + {0, 1, 2}] = {sum or mean, min, max} of column col < ncol of A [n x ld] (n >= 1)
    void run(sb_ctx *ctx, const double *A, u32 ld, u32 ncol, u64 n, const double *c, int mean, double *out) {
        const u64 nch = (n + TS_CHUNK - 1) / TS_CHUNK;
        k_ts_part<<<ts_grid(ctx, nch * ncol, 128), 128, 0, ctx->stream>>>(A, ld, ncol, n, c, sum.p, mn.p, mx.p);
        k_ts_fin<<<cdiv(ncol, 32), 32, 0, ctx->stream>>>(sum.p, mn.p, mx.p, nch, ncol, n, mean, out);
        count_launch(ctx);
        count_launch(ctx);
    }
};

// ---------------------------------------------------------------- affinities
// thread per element of X [n x dim]: X - mean (st[3 c] the column means), the largest |x| into *amax (positive doubles order as
// their bits)
__global__ void k_ts_center_cols(double *__restrict__ X, u64 n, u32 dim, const double *__restrict__ st, ull *__restrict__ amax) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < n * dim; x += (u64)gridDim.x * blockDim.x) {
        const double v = X[x] - st[3 * (x % dim)];
        X[x] = v;
        atomicMax(amax, (ull)__double_as_longlong(fabs(v)));
    }
}
__global__ void k_ts_scale(double *__restrict__ X, u64 count, const ull *__restrict__ amax) {
    const double m = __longlong_as_double((long long)*amax);
    if (!(m > 0.0)) return;
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (u64)gridDim.x * blockDim.x) X[x] = X[x] / m;
}

// thread per row: bhtsne's beta search on D = d d of the listed slots, then the row divided by sum_P; pc[s] (0 at padding), beta[i]
// (the beta that gave the row), the forward key (i << 32 | j, value: the slot) and the transposed key (j << 32 | i, value: the slot
// | TS_TAG); all-ones keys at padding
__global__ void k_ts_beta(const double *__restrict__ d, const u32 *__restrict__ nbr, u64 n, u32 k, double log_perp, double *__restrict__ pc,
                          double *__restrict__ beta_out, u64 *__restrict__ keys, u64 *__restrict__ vals) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const double *di = d + i * k;
        const u32 *ri = nbr + i * k;
        double beta = 1.0, lo = -DBL_MAX, hi = DBL_MAX, used = 1.0, sum_P = DBL_MIN;
        for (int it = 0; it < 200; it++) {
            sum_P = DBL_MIN;
            double H = 0.0;
            for (u32 t = 0; t < k; t++) {
                if (ri[t] == TS_PAD) continue;
                const double D = di[t] * di[t], p = exp(-(beta * D));
                sum_P = sum_P + p;
                H = H + beta * (D * p);
            }
            H = H / sum_P + log(sum_P);
            used = beta;
            const double hd = H - log_perp;
            if (hd < 1e-5 && -hd < 1e-5) break;
            if (hd > 0.0) {
                lo = beta;
                beta = (hi == DBL_MAX || hi == -DBL_MAX) ? beta * 2.0 : (beta + hi) / 2.0;
            } else {
                hi = beta;
                beta = (lo == -DBL_MAX || lo == DBL_MAX) ? beta / 2.0 : (beta + lo) / 2.0;
            }
        }
        beta_out[i] = used;
        for (u32 t = 0; t < k; t++) {
            const u64 s = i * k + t;
            const u32 j = ri[t];
            if (j == TS_PAD) {
                pc[s] = 0.0;
                keys[2 * s] = keys[2 * s + 1] = ~0ull;
                vals[2 * s] = vals[2 * s + 1] = 0;
                continue;
            }
            pc[s] = exp(-(used * (di[t] * di[t]))) / sum_P;
            keys[2 * s] = (i << 32) | j;
            vals[2 * s] = s;
            keys[2 * s + 1] = ((u64)j << 32) | i;
            vals[2 * s + 1] = s | TS_TAG;
        }
    }
}

// thread per sorted entry: the first entry of a pair adds a = P_i|j and b = P_j|i (0 when not listed) as a + b; zeros and the
// all-ones keys of padding dropped
__global__ void k_ts_join(const u64 *__restrict__ keys, const u64 *__restrict__ vals, u64 count, const double *__restrict__ pc, double *__restrict__ out,
                          char *__restrict__ keep) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (u64)gridDim.x * blockDim.x) {
        keep[x] = 0;
        out[x] = 0.0;
        if ((x && keys[x] == keys[x - 1]) || keys[x] == ~0ull) continue;
        double a = 0.0, b = 0.0;
        for (u64 y = x; y < count && y < x + 2 && keys[y] == keys[x]; y++) {
            const u64 v = vals[y];
            if (v & TS_TAG) b = pc[v & ~TS_TAG];
            else a = pc[v];
        }
        const double r = a + b;
        out[x] = r;
        keep[x] = r > 0.0;
    }
}
__global__ void k_ts_divide(double *__restrict__ v, u64 count, const double *__restrict__ tot) {
    const double t = *tot;
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (u64)gridDim.x * blockDim.x) v[x] = v[x] / t;
}

// X [n x dim], nbr [n x k] on the device (X is scaled in place) -> P (g), beta (device)
static int ts_affinities(sb_ctx *ctx, double *X, const u32 *nbr, u64 n, u32 dim, u32 k, double perplexity, UmGraph &g, DevBuf<double> &beta,
                         const char *fn) {
    TraceScope tr(ctx, "tsne: affinities");
    const u64 nk = n * k, np = 2 * nk;
    TsSum ts;
    DevBuf<double> st, d, pc;
    DevBuf<ull> amax;
    DevBuf<int> err;
    DevBuf<u64> keys, vals;
    SB_TRY(ts.init(n, dim));
    SB_TRY(st.alloc(3 * (u64)dim));
    SB_TRY(amax.alloc(1));
    SB_TRY(err.alloc(1));
    SB_TRY(d.alloc(nk));
    SB_TRY(pc.alloc(nk));
    SB_TRY(beta.alloc(n));
    SB_TRY(keys.alloc(np));
    SB_TRY(vals.alloc(np));
    SB_CUDA(cudaMemsetAsync(amax.p, 0, sizeof(ull), ctx->stream));
    SB_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), ctx->stream));
    ts.run(ctx, X, dim, dim, n, nullptr, 1, st.p);
    k_ts_center_cols<<<ts_grid(ctx, n * dim, 256), 256, 0, ctx->stream>>>(X, n, dim, st.p, amax.p);
    k_ts_scale<<<ts_grid(ctx, n * dim, 256), 256, 0, ctx->stream>>>(X, n * dim, amax.p);
    k_um_dist<<<ts_grid(ctx, nk, 256), 256, 0, ctx->stream>>>(X, nbr, n, dim, k, d.p, err.p);
    k_ts_beta<<<ts_grid(ctx, n, 128), 128, 0, ctx->stream>>>(d.p, nbr, n, k, log(perplexity), pc.p, beta.p, keys.p, vals.p);
    for (int q = 0; q < 4; q++) count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    int herr = 0;
    SB_CUDA(cudaMemcpyAsync(&herr, err.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (herr)
        return sb_fail(SB_ERR_INVALID_ARG, "%s: invalid neighbour lists:%s%s%s%s", fn, herr & 1 ? " an index >= n" : "", herr & 2 ? " a self index" : "",
                       herr & 4 ? " a duplicate in a row" : "", herr & 8 ? " padding before the row end" : "");
    d.release();
    DevBuf<double> sym, gv;
    DevBuf<char> keep;
    DevBuf<u64> gk, num;
    SB_TRY(sort_pairs(ctx, keys, vals, np));
    SB_TRY(sym.alloc(np));
    SB_TRY(keep.alloc(np));
    SB_TRY(gk.alloc(np));
    SB_TRY(gv.alloc(np));
    SB_TRY(num.alloc(1));
    k_ts_join<<<ts_grid(ctx, np, 256), 256, 0, ctx->stream>>>(keys.p, vals.p, np, pc.p, sym.p, keep.p);
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    SB_TRY(um_select(ctx, keys.p, keep.p, gk.p, np, num.p));
    SB_TRY(um_select(ctx, sym.p, keep.p, gv.p, np, num.p));
    u64 nnz = 0;
    SB_CUDA(cudaMemcpyAsync(&nnz, num.p, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    g.n = n;
    g.nnz = nnz;
    SB_TRY(um_rows_from_keys(ctx, gk.p, g));
    if (nnz) {  // the total in CSR order, chunked
        TsSum tt;
        SB_TRY(tt.init(nnz, 1));
        tt.run(ctx, gv.p, 1, 1, nnz, nullptr, 0, st.p);
        k_ts_divide<<<ts_grid(ctx, nnz, 256), 256, 0, ctx->stream>>>(gv.p, nnz, st.p);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
    }
    g.w.swap(gv);
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- the tree
// 32 bits of v spread to the even bits of a 64-bit word
__device__ __forceinline__ u64 ts_spread(u64 v) {
    v = (v | (v << 16)) & 0x0000FFFF0000FFFFull;
    v = (v | (v << 8)) & 0x00FF00FF00FF00FFull;
    v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v << 2)) & 0x3333333333333333ull;
    v = (v | (v << 1)) & 0x5555555555555555ull;
    return v;
}
// the root box from st (mean, min, max per axis): centre = mean, half-width = max(max - mean, mean - min) + 1e-5
__device__ __forceinline__ void ts_box(const double *st, int a, double &lo, double &hw) {
    const double m = st[3 * a];
    hw = fmax(st[3 * a + 2] - m, m - st[3 * a + 1]) + 1e-5;
    lo = m - hw;
}
// y to 32 bits in [lo, lo + 2 hw): floor((y - lo) / (hw + hw) 2^32), clamped
__device__ __forceinline__ u64 ts_quant(double y, double lo, double hw) {
    const double v = (y - lo) / (hw + hw) * 4294967296.0;
    return v >= 4294967295.0 ? 0xFFFFFFFFull : (v > 0.0 ? (u64)v : 0ull);
}
// thread per point: key = x bits at the odd positions (bit 63 the top x bit), y bits at the even; value = the point
__global__ void k_ts_codes(const double *__restrict__ Y, u64 n, const double *__restrict__ st, u64 *__restrict__ keys, u64 *__restrict__ vals) {
    double lx, hx, ly, hy;
    ts_box(st, 0, lx, hx);
    ts_box(st, 1, ly, hy);
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        keys[i] = (ts_spread(ts_quant(Y[2 * i], lx, hx)) << 1) | ts_spread(ts_quant(Y[2 * i + 1], ly, hy));
        vals[i] = i;
    }
}
__global__ void k_ts_runs(const u64 *__restrict__ keys, u64 n, u32 *__restrict__ flag) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (u64)gridDim.x * blockDim.x) flag[x] = x == 0 || keys[x] != keys[x - 1];
}
// thread per sorted position (lid: the inclusive scan of the run flags): run starts, the distinct codes, their number m
__global__ void k_ts_leaves(const u64 *__restrict__ keys, const u32 *__restrict__ flag, const u32 *__restrict__ lid, u64 n, u32 *__restrict__ start,
                            u64 *__restrict__ lkey, u32 *__restrict__ m) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (u64)gridDim.x * blockDim.x) {
        const u32 l = lid[x] - 1;
        if (flag[x]) {
            start[l] = (u32)x;
            lkey[l] = keys[x];
        }
        if (x == n - 1) {
            *m = l + 1;
            start[l + 1] = (u32)n;
        }
    }
}
__device__ __forceinline__ int ts_delta(const u64 *k, long long m, long long i, long long j) {
    return (j < 0 || j >= m) ? -1 : __clzll(k[i] ^ k[j]);
}
// Karras 2012 over the m distinct codes: thread per internal node i < m - 1 (node 0 the root); children with TS_LEAF for leaves,
// the parents, and the common prefix length of the node's codes
__global__ void k_ts_karras(const u64 *__restrict__ k, const u32 *__restrict__ mp, u32 *__restrict__ child, u32 *__restrict__ par_int,
                            u32 *__restrict__ par_leaf, u32 *__restrict__ pref) {
    const long long m = *mp;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m - 1; i += (long long)gridDim.x * blockDim.x) {
        const int d = ts_delta(k, m, i, i + 1) - ts_delta(k, m, i, i - 1) > 0 ? 1 : -1;
        const int dmin = ts_delta(k, m, i, i - d);
        long long lmax = 2;
        while (ts_delta(k, m, i, i + lmax * d) > dmin) lmax *= 2;
        long long l = 0;
        for (long long t = lmax / 2; t >= 1; t /= 2)
            if (ts_delta(k, m, i, i + (l + t) * d) > dmin) l += t;
        const long long j = i + l * d;
        const int dn = ts_delta(k, m, i, j);
        long long s = 0;
        for (long long div = 2;; div *= 2) {
            const long long t = (l + div - 1) / div;
            if (ts_delta(k, m, i, i + (s + t) * d) > dn) s += t;
            if (t <= 1) break;
        }
        const long long g = i + s * d + (d < 0 ? -1 : 0), lo = i < j ? i : j, hi = i < j ? j : i;
        const u32 left = lo == g ? (TS_LEAF | (u32)g) : (u32)g, right = hi == g + 1 ? (TS_LEAF | (u32)(g + 1)) : (u32)(g + 1);
        child[2 * i] = left;
        child[2 * i + 1] = right;
        if (left & TS_LEAF) par_leaf[g] = (u32)i;
        else par_int[g] = (u32)i;
        if (right & TS_LEAF) par_leaf[g + 1] = (u32)i;
        else par_int[g + 1] = (u32)i;
        pref[i] = (u32)dn;
    }
}
// thread per leaf: count and sum of y over its run in sorted order (from 0); then up the tree, the second thread to arrive at a node
// writes it as left + right
__global__ void k_ts_sums(const double *__restrict__ Y, const u64 *__restrict__ perm, const u32 *__restrict__ start, const u32 *__restrict__ mp,
                          const u32 *__restrict__ child, const u32 *__restrict__ par_int, const u32 *__restrict__ par_leaf, u32 *visits, u32 *cnt_l,
                          double *sum_l, u32 *cnt_i, double *sum_i) {
    const u32 m = *mp;
    for (u64 l = (u64)blockIdx.x * blockDim.x + threadIdx.x; l < m; l += (u64)gridDim.x * blockDim.x) {
        const u32 a = start[l], b = start[l + 1];
        double sx = 0.0, sy = 0.0;
        for (u32 x = a; x < b; x++) {
            const u64 i = perm[x];
            sx = sx + Y[2 * i];
            sy = sy + Y[2 * i + 1];
        }
        cnt_l[l] = b - a;
        sum_l[2 * l] = sx;
        sum_l[2 * l + 1] = sy;
        if (m == 1) continue;
        u32 node = par_leaf[l];
        while (true) {
            __threadfence();
            if (atomicAdd(&visits[node], 1u) == 0) break;
            __threadfence();
            const u32 L = child[2 * node], R = child[2 * node + 1];
            const volatile u32 *vc_l = cnt_l, *vc_i = cnt_i;
            const volatile double *vs_l = sum_l, *vs_i = sum_i;
            const u32 cl = (L & TS_LEAF) ? vc_l[L & ~TS_LEAF] : vc_i[L], cr = (R & TS_LEAF) ? vc_l[R & ~TS_LEAF] : vc_i[R];
            double s[2];
            for (int c = 0; c < 2; c++) {
                const double u = (L & TS_LEAF) ? vs_l[2 * (L & ~TS_LEAF) + c] : vs_i[2 * L + c];
                const double v = (R & TS_LEAF) ? vs_l[2 * (R & ~TS_LEAF) + c] : vs_i[2 * R + c];
                s[c] = u + v;
            }
            cnt_i[node] = cl + cr;
            sum_i[2 * node] = s[0];
            sum_i[2 * node + 1] = s[1];
            if (node == 0) break;
            node = par_int[node];
        }
    }
}

struct TsTree {
    const u64 *perm;         // [n] points in code order
    const u32 *lid;          // [n] leaf of sorted position x, plus one
    const u32 *m;            // the number of leaves (device)
    const u32 *child, *pref; // internal nodes
    const u32 *cnt_l, *cnt_i;
    const double *sum_l, *sum_i;
    const double *st;        // the root box
};

// the Barnes-Hut walk of point i (sorted position x): neg (the unnormalised repulsion) and its q sum
__device__ __forceinline__ void ts_walk(const TsTree &t, u64 x, double yx, double yy, double theta, double &nx, double &ny, double &q) {
    double lx, hx, ly, hy;
    ts_box(t.st, 0, lx, hx);
    ts_box(t.st, 1, ly, hy);
    const u32 m = *t.m, mine = t.lid[x] - 1;
    u32 stack[TS_STACK];
    int sp = 0;
    stack[sp++] = m == 1 ? TS_LEAF : 0u;
    nx = ny = q = 0.0;
    while (sp) {
        const u32 node = stack[--sp];
        double cnt, cx, cy;
        if (node & TS_LEAF) {
            const u32 l = node & ~TS_LEAF;
            u32 c = t.cnt_l[l];
            double sx = t.sum_l[2 * l], sy = t.sum_l[2 * l + 1];
            if (l == mine) {  // the point's own leaf, without the point
                if (c == 1) continue;
                c -= 1;
                sx = sx - yx;
                sy = sy - yy;
            }
            cnt = (double)c;
            cx = sx / cnt;
            cy = sy / cnt;
        } else {
            cnt = (double)t.cnt_i[node];
            cx = t.sum_i[2 * node] / cnt;
            cy = t.sum_i[2 * node + 1] / cnt;
        }
        const double bx = yx - cx, by = yy - cy;
        const double D = bx * bx + by * by;
        if (!(node & TS_LEAF)) {
            const u32 p = t.pref[node], ex = (p + 1) >> 1, ey = p >> 1;  // bits fixed per axis: x takes the odd positions from the top
            const double wx = hx * __longlong_as_double((long long)(1023 - ex) << 52), wy = hy * __longlong_as_double((long long)(1023 - ey) << 52);
            if (!(fmax(wx, wy) / sqrt(D) < theta)) {
                stack[sp++] = t.child[2 * node + 1];
                stack[sp++] = t.child[2 * node];
                continue;
            }
        }
        const double qq = 1.0 / (1.0 + D);
        double mult = cnt * qq;
        q = q + mult;
        mult = mult * qq;
        nx = nx + mult * bx;
        ny = ny + mult * by;
    }
}

// thread per sorted position: pos (attractive, e P_ij over the CSR row in column order) and neg (the walk) of the point, and q
__global__ void __launch_bounds__(128) k_ts_forces(TsTree t, const double *__restrict__ Y, u64 n, const u64 *__restrict__ ptr, const u32 *__restrict__ idx,
                                                   const double *__restrict__ P, double ex, double theta, double *__restrict__ pos,
                                                   double *__restrict__ neg, double *__restrict__ qs) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < n; x += (u64)gridDim.x * blockDim.x) {
        const u64 i = t.perm[x];
        const double yx = Y[2 * i], yy = Y[2 * i + 1];
        double px = 0.0, py = 0.0;
        for (u64 e = ptr[i]; e < ptr[i + 1]; e++) {
            const u32 j = idx[e];
            const double bx = yx - Y[2 * (u64)j], by = yy - Y[2 * (u64)j + 1];
            double D = 1.0 + bx * bx;
            D = D + by * by;
            const double w = (ex * P[e]) / D;
            px = px + w * bx;
            py = py + w * by;
        }
        double nx, ny, q;
        ts_walk(t, x, yx, yy, theta, nx, ny, q);
        pos[2 * i] = px;
        pos[2 * i + 1] = py;
        neg[2 * i] = nx;
        neg[2 * i + 1] = ny;
        qs[i] = q;
    }
}

__global__ void k_ts_fill(double *__restrict__ v, u64 count, double x) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (u64)gridDim.x * blockDim.x) v[i] = x;
}
__device__ __forceinline__ double ts_sign(double v) { return v == 0.0 ? 0.0 : (v < 0.0 ? -1.0 : 1.0); }
// thread per coordinate: dY = pos - neg / sum_Q; bhtsne's gains; uY = mom uY - (eta gains) dY; Y += uY
__global__ void k_ts_update(double *__restrict__ Y, double *__restrict__ uY, double *__restrict__ gains, const double *__restrict__ pos,
                            const double *__restrict__ neg, const double *__restrict__ sq, u64 count, double mom, double eta) {
    const double sum_Q = *sq;
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (u64)gridDim.x * blockDim.x) {
        const double dY = pos[x] - neg[x] / sum_Q, u = uY[x];
        double g = gains[x];
        g = ts_sign(dY) != ts_sign(u) ? g + 0.2 : g * 0.8;
        if (g < 0.01) g = 0.01;
        const double nu = mom * u - (eta * g) * dY;
        gains[x] = g;
        uY[x] = nu;
        Y[x] = Y[x] + nu;
    }
}
__global__ void k_ts_center(double *__restrict__ Y, u64 count, const double *__restrict__ st) {
    const double mx = st[0], my = st[3];
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < count; x += (u64)gridDim.x * blockDim.x) Y[x] = Y[x] - ((x & 1) ? my : mx);
}
// thread per row: bhtsne's evaluateError terms P log((P + FLT_MIN) / (Q + FLT_MIN)), Q = (1 / (1 + |y_i - y_j|^2)) / sum_Q
__global__ void k_ts_kl(const double *__restrict__ Y, u64 n, const u64 *__restrict__ ptr, const u32 *__restrict__ idx, const double *__restrict__ P,
                        const double *__restrict__ sq, double *__restrict__ out) {
    const double sum_Q = *sq;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        double c = 0.0;
        for (u64 e = ptr[i]; e < ptr[i + 1]; e++) {
            const u64 j = idx[e];
            const double bx = Y[2 * i] - Y[2 * j], by = Y[2 * i + 1] - Y[2 * j + 1];
            const double Q = (1.0 / (1.0 + (bx * bx + by * by))) / sum_Q;
            c = c + P[e] * log((P[e] + (double)FLT_MIN) / (Q + (double)FLT_MIN));
        }
        out[i] = c;
    }
}

// ---------------------------------------------------------------- start positions
// mode 0 (PCA): A's first two columns / sd * 1e-4 (sd of column 0, st[0]); 1: N(0, 1e-4^2) by Box-Muller from the counter hash;
// 2: A as given
__global__ void k_ts_init(const double *__restrict__ A, u64 n, u32 ld, int mode, const double *__restrict__ sd, u64 key, double *__restrict__ Y) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        if (mode == 0) {
            const double s = *sd;
            Y[2 * i] = A[i * ld] / s * 1e-4;
            Y[2 * i + 1] = A[i * ld + 1] / s * 1e-4;
        } else if (mode == 1) {
            const double u1 = (double)((um_mix64(key ^ (2 * i)) >> 11) + 1) * 0x1p-53, u2 = (double)(um_mix64(key ^ (2 * i + 1)) >> 11) * 0x1p-53;
            const double r = sqrt(-2.0 * log(u1)), a = 6.283185307179586 * u2;
            Y[2 * i] = 1e-4 * (r * cos(a));
            Y[2 * i + 1] = 1e-4 * (r * sin(a));
        } else {
            Y[2 * i] = A[i * ld];
            Y[2 * i + 1] = A[i * ld + 1];
        }
    }
}
__global__ void k_ts_sd(const double *__restrict__ st, u64 n, double *__restrict__ sd) { *sd = sqrt(st[0] / (double)n); }

// ---------------------------------------------------------------- options
struct TsOpts {
    double perplexity, theta, lr, exag;
    u32 max_iter, stop_lying, mom_switch, nc, init;
    u64 seed;
};

static int ts_opts(const sb_tsne_opts *o, TsOpts &out, const char *fn) {
    out = TsOpts{30.0, 0.5, 200.0, 12.0, 1000, 250, 250, 2, SB_TSNE_INIT_PCA, 0};
    if (!o) return SB_OK;
    out = TsOpts{o->perplexity, o->theta, o->learning_rate, o->early_exaggeration, o->max_iter, o->stop_lying_iter, o->mom_switch_iter, o->n_components,
                 o->init, o->seed};
    if (!(out.perplexity > 0.0) || !std::isfinite(out.perplexity)) return sb_fail(SB_ERR_INVALID_ARG, "%s: perplexity must be finite and > 0", fn);
    if (!(out.theta >= 0.0) || !std::isfinite(out.theta)) return sb_fail(SB_ERR_INVALID_ARG, "%s: theta must be finite and >= 0", fn);
    if (!(out.lr >= 0.0) || !std::isfinite(out.lr)) return sb_fail(SB_ERR_INVALID_ARG, "%s: learning_rate must be finite and >= 0", fn);
    if (!(out.exag > 0.0) || !std::isfinite(out.exag)) return sb_fail(SB_ERR_INVALID_ARG, "%s: early_exaggeration must be finite and > 0", fn);
    if (out.init > SB_TSNE_INIT_USER) return sb_fail(SB_ERR_INVALID_ARG, "%s: init must be SB_TSNE_INIT_PCA, _RANDOM or _USER", fn);
    if (out.nc != 2) return sb_fail(SB_ERR_UNSUPPORTED, "%s: n_components must be 2", fn);
    return SB_OK;
}

// bhtsne's checks of perplexity against n and k, and the shape limits shared with UMAP
static int ts_knn_args(uint64_t n, uint32_t dim, uint32_t k, double perplexity, const char *fn) {
    if (dim == 0) return sb_fail(SB_ERR_INVALID_ARG, "%s: dim must be >= 1", fn);
    if ((double)n - 1.0 < 3.0 * perplexity) return sb_fail(SB_ERR_INVALID_ARG, "%s: perplexity too large for the number of points (n - 1 < 3 perplexity)", fn);
    const u64 K = (u64)std::floor(3.0 * perplexity), need = std::min<u64>(n - 1, K);
    if (k < need) return sb_fail(SB_ERR_INVALID_ARG, "%s: k = %u is below min(n - 1, floor(3 perplexity)) = %llu", fn, k, (unsigned long long)need);
    if (k > TS_MAX_K) return sb_fail(SB_ERR_UNSUPPORTED, "%s: k must be <= %d", fn, TS_MAX_K);
    if (n >= 0x7FFFFFFFull || n * k >= ((u64)1 << 28)) return sb_fail(SB_ERR_UNSUPPORTED, "%s: n x k must be below 2^28", fn);
    return SB_OK;
}

static int ts_user_init(const double *init, u64 rows, const char *fn) {
    if (rows && !init) return sb_fail(SB_ERR_INVALID_ARG, "%s: init must hold n x 2 values", fn);
    for (u64 x = 0; x < 2 * rows; x++)
        if (!std::isfinite(init[x])) return sb_fail(SB_ERR_INVALID_ARG, "%s: init values must be finite", fn);
    return SB_OK;
}

// start positions Y [n x 2] from A [n x ld] (mode PCA scales its first two columns, USER takes them, RANDOM ignores A)
static int ts_init(sb_ctx *ctx, const double *A, u64 n, u32 ld, const TsOpts &o, DevBuf<double> &Y, const char *fn) {
    SB_TRY(Y.alloc(2 * n));
    if (!n) return SB_OK;
    const int mode = o.init == SB_TSNE_INIT_PCA ? 0 : o.init == SB_TSNE_INIT_RANDOM ? 1 : 2;
    DevBuf<double> st, sd;
    SB_TRY(st.alloc(6));
    SB_TRY(sd.alloc(1));
    if (mode == 0) {  // the population sd of column 0: the mean, then the squared deviations, both in chunked order
        TsSum ts;
        SB_TRY(ts.init(n, 1));
        ts.run(ctx, A, ld, 1, n, nullptr, 1, st.p);
        ts.run(ctx, A, ld, 1, n, st.p, 0, st.p + 3);
        k_ts_sd<<<1, 1, 0, ctx->stream>>>(st.p + 3, n, sd.p);
        count_launch(ctx);
        double h = 0.0;
        SB_CUDA(cudaMemcpyAsync(&h, sd.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        if (!(h > 0.0) || !std::isfinite(h)) return sb_fail(SB_ERR_INVALID_ARG, "%s: the pca start needs a first score column that is finite and not constant", fn);
    }
    k_ts_init<<<ts_grid(ctx, n, 256), 256, 0, ctx->stream>>>(A, n, ld, mode, sd.p, um_mix64(um_mix64(o.seed) ^ ~0ull), Y.p);
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

// ---------------------------------------------------------------- layout
// the iterations on P (g) from the start Y -> Y; info
static int ts_layout(sb_ctx *ctx, const UmGraph &g, DevBuf<double> &Y, const TsOpts &o, sb_tsne_info *info) {
    const u64 n = g.n;
    const double eta = o.lr > 0.0 ? o.lr : std::max((double)n / (4.0 * o.exag), 50.0);
    info->kl_divergence = 0.0;
    info->learning_rate = eta;
    info->nnz = g.nnz;
    info->n_iter = o.max_iter;
    info->reserved = 0;
    if (!n) return SB_OK;
    TraceScope tr(ctx, "tsne: layout");
    DevBuf<double> uY, gains, pos, neg, qs, st, sq, sum_l, sum_i;
    DevBuf<u64> keys, vals, skeys, perm, lkey;
    DevBuf<u32> flag, lid, start, m, child, par_int, par_leaf, pref, visits, cnt_l, cnt_i;
    TsSum ty, tq;
    const u64 ni = std::max<u64>(1, n - 1);
    SB_TRY(uY.alloc(2 * n));
    SB_TRY(gains.alloc(2 * n));
    SB_TRY(pos.alloc(2 * n));
    SB_TRY(neg.alloc(2 * n));
    SB_TRY(qs.alloc(n));
    SB_TRY(st.alloc(6));
    SB_TRY(sq.alloc(3));
    SB_TRY(sum_l.alloc(2 * n));
    SB_TRY(sum_i.alloc(2 * ni));
    SB_TRY(keys.alloc(n));
    SB_TRY(vals.alloc(n));
    SB_TRY(skeys.alloc(n));
    SB_TRY(perm.alloc(n));
    SB_TRY(lkey.alloc(n));
    SB_TRY(flag.alloc(n));
    SB_TRY(lid.alloc(n));
    SB_TRY(start.alloc(n + 1));
    SB_TRY(m.alloc(1));
    SB_TRY(child.alloc(2 * ni));
    SB_TRY(par_int.alloc(ni));
    SB_TRY(par_leaf.alloc(n));
    SB_TRY(pref.alloc(ni));
    SB_TRY(visits.alloc(ni));
    SB_TRY(cnt_l.alloc(n));
    SB_TRY(cnt_i.alloc(ni));
    SB_TRY(ty.init(n, 2));
    SB_TRY(tq.init(n, 1));
    size_t scan_bytes = 0;
    SB_CUDA(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, flag.p, lid.p, n, ctx->stream));
    DevBuf<char> scan_tmp;
    SB_TRY(scan_tmp.alloc(scan_bytes));
    // the codes are sorted into fixed buffers (a stable radix sort, as sort_pairs): the loop allocates nothing
    size_t sort_bytes = 0;
    SB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, keys.p, skeys.p, vals.p, perm.p, n, 0, 64, ctx->stream));
    DevBuf<char> sort_tmp;
    SB_TRY(sort_tmp.alloc(sort_bytes));
    SB_CUDA(cudaMemsetAsync(uY.p, 0, 2 * n * sizeof(double), ctx->stream));
    k_ts_fill<<<ts_grid(ctx, 2 * n, 256), 256, 0, ctx->stream>>>(gains.p, 2 * n, 1.0);
    count_launch(ctx);
    const int gp = ts_grid(ctx, n, 256);
    // the tree of the current Y and the forces on it (neg, q per point; pos with exaggeration ex)
    auto tree_and_forces = [&](double ex) -> int {
        {
            TraceScope tt(ctx, "tsne: tree");
            ty.run(ctx, Y.p, 2, 2, n, nullptr, 1, st.p);
            k_ts_codes<<<gp, 256, 0, ctx->stream>>>(Y.p, n, st.p, keys.p, vals.p);
            count_launch(ctx);
            SB_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp.p, sort_bytes, keys.p, skeys.p, vals.p, perm.p, n, 0, 64, ctx->stream));
            count_launch(ctx, false);
            k_ts_runs<<<gp, 256, 0, ctx->stream>>>(skeys.p, n, flag.p);
            count_launch(ctx);
            SB_CUDA(cub::DeviceScan::InclusiveSum(scan_tmp.p, scan_bytes, flag.p, lid.p, n, ctx->stream));
            count_launch(ctx, false);
            k_ts_leaves<<<gp, 256, 0, ctx->stream>>>(skeys.p, flag.p, lid.p, n, start.p, lkey.p, m.p);
            k_ts_karras<<<ts_grid(ctx, ni, 256), 256, 0, ctx->stream>>>(lkey.p, m.p, child.p, par_int.p, par_leaf.p, pref.p);
            SB_CUDA(cudaMemsetAsync(visits.p, 0, ni * sizeof(u32), ctx->stream));
            k_ts_sums<<<gp, 256, 0, ctx->stream>>>(Y.p, perm.p, start.p, m.p, child.p, par_int.p, par_leaf.p, visits.p, cnt_l.p, sum_l.p, cnt_i.p, sum_i.p);
            for (int q = 0; q < 3; q++) count_launch(ctx);
        }
        TraceScope tf(ctx, "tsne: forces");
        TsTree t{perm.p, lid.p, m.p, child.p, pref.p, cnt_l.p, cnt_i.p, sum_l.p, sum_i.p, st.p};
        k_ts_forces<<<ts_grid(ctx, n, 128), 128, 0, ctx->stream>>>(t, Y.p, n, g.ptr.p, g.idx.p, g.w.p, ex, o.theta, pos.p, neg.p, qs.p);
        count_launch(ctx);
        tq.run(ctx, qs.p, 1, 1, n, nullptr, 0, sq.p);
        SB_CUDA(cudaGetLastError());
        return SB_OK;
    };
    for (u32 it = 0; it < o.max_iter; it++) {
        // bhtsne divides P by the exaggeration and switches the momentum after the update of iterations stop_lying_iter and
        // mom_switch_iter: those iterations still use the first values
        SB_TRY(tree_and_forces(it <= o.stop_lying ? o.exag : 1.0));
        TraceScope tu(ctx, "tsne: update");
        k_ts_update<<<ts_grid(ctx, 2 * n, 256), 256, 0, ctx->stream>>>(Y.p, uY.p, gains.p, pos.p, neg.p, sq.p, 2 * n, it <= o.mom_switch ? 0.5 : 0.8, eta);
        ty.run(ctx, Y.p, 2, 2, n, nullptr, 1, st.p);
        k_ts_center<<<ts_grid(ctx, 2 * n, 256), 256, 0, ctx->stream>>>(Y.p, 2 * n, st.p);
        count_launch(ctx);
        count_launch(ctx);
    }
    // bhtsne's evaluateError: sum_Q from the walk on the final Y, the KL terms per row, summed in chunked order
    SB_TRY(tree_and_forces(1.0));
    k_ts_kl<<<ts_grid(ctx, n, 128), 128, 0, ctx->stream>>>(Y.p, n, g.ptr.p, g.idx.p, g.w.p, sq.p, qs.p);
    count_launch(ctx);
    tq.run(ctx, qs.p, 1, 1, n, nullptr, 0, sq.p);
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaMemcpyAsync(&info->kl_divergence, sq.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

static int ts_copy_out(sb_ctx *ctx, const DevBuf<double> &Y, u64 first, u64 count, double *out) {
    if (!count) return SB_OK;
    SB_CUDA(cudaMemcpyAsync(out, Y.p + 2 * first, 2 * count * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- entry points
extern "C" int sb_tsne_affinities(sb_ctx *ctx, const double *X, const uint32_t *nbr, uint64_t n, uint32_t dim, uint32_t k, const sb_tsne_opts *opts,
                                  uint64_t *indptr, uint32_t *indices, double *P, uint64_t *nnz, double *beta) {
    if (!ctx || !indptr || !nnz || (n && k && (!indices || !P))) return sb_fail(SB_ERR_INVALID_ARG, "sb_tsne_affinities: NULL argument");
    TsOpts o;
    SB_TRY(ts_opts(opts, o, "sb_tsne_affinities"));
    if (n && (!X || !nbr)) return sb_fail(SB_ERR_INVALID_ARG, "sb_tsne_affinities: NULL argument");
    SB_TRY(ts_knn_args(n, dim, k, o.perplexity, "sb_tsne_affinities"));
    SB_ENTER(ctx);
    DevBuf<double> dX, db;
    DevBuf<u32> dn;
    SB_TRY(dX.alloc(n * dim));
    SB_TRY(dn.alloc(n * k));
    SB_CUDA(cudaMemcpyAsync(dX.p, X, n * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(dn.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    UmGraph g;
    SB_TRY(ts_affinities(ctx, dX.p, dn.p, n, dim, k, o.perplexity, g, db, "sb_tsne_affinities"));
    SB_CUDA(cudaMemcpyAsync(indptr, g.ptr.p, (n + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    if (g.nnz) {
        SB_CUDA(cudaMemcpyAsync(indices, g.idx.p, g.nnz * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(P, g.w.p, g.nnz * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (beta) SB_CUDA(cudaMemcpyAsync(beta, db.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    *nnz = g.nnz;
    return SB_OK;
}

extern "C" int sb_tsne_layout(sb_ctx *ctx, uint64_t n, const uint64_t *indptr, const uint32_t *indices, const double *P, const double *init,
                              const sb_tsne_opts *opts, double *out, sb_tsne_info *info) {
    if (!ctx || !indptr || !info || (n && !out)) return sb_fail(SB_ERR_INVALID_ARG, "sb_tsne_layout: NULL argument");
    TsOpts o;
    SB_TRY(ts_opts(opts, o, "sb_tsne_layout"));
    SB_TRY(um_csr_host_check(n, indptr, indices, P, "sb_tsne_layout"));
    if (o.init != SB_TSNE_INIT_RANDOM) SB_TRY(ts_user_init(init, n, "sb_tsne_layout"));
    SB_ENTER(ctx);
    UmGraph g;
    SB_TRY(um_csr_upload(ctx, n, indptr, indices, P, g, "sb_tsne_layout", "tsne: csr validation"));
    DevBuf<double> dA, Y;
    SB_TRY(dA.alloc(2 * n));
    if (n && o.init != SB_TSNE_INIT_RANDOM) SB_CUDA(cudaMemcpyAsync(dA.p, init, 2 * n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    SB_TRY(ts_init(ctx, dA.p, n, 2, o, Y, "sb_tsne_layout"));
    SB_TRY(ts_layout(ctx, g, Y, o, info));
    return ts_copy_out(ctx, Y, 0, n, out);
}

extern "C" int sb_tsne(sb_ctx *ctx, const double *X, const uint32_t *nbr, uint64_t n_local, uint32_t dim, uint32_t k, const sb_tsne_opts *opts,
                       const double *init, double *out, sb_tsne_info *info) {
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "sb_tsne: NULL argument");
    TsOpts o;
    int rc = (!info || (n_local && !out) || (n_local && (!X || !nbr))) ? sb_fail(SB_ERR_INVALID_ARG, "sb_tsne: NULL argument") : SB_OK;
    if (rc == SB_OK) rc = ts_opts(opts, o, "sb_tsne");
    if (rc == SB_OK && dim == 0) rc = sb_fail(SB_ERR_INVALID_ARG, "sb_tsne: dim must be >= 1");
    if (rc == SB_OK && dim < 2 && o.init == SB_TSNE_INIT_PCA) rc = sb_fail(SB_ERR_INVALID_ARG, "sb_tsne: pca init needs dim >= 2");
    if (rc == SB_OK && o.init == SB_TSNE_INIT_USER) rc = ts_user_init(init, n_local, "sb_tsne");
    SB_ENTER(ctx);
    SB_TRY(agree_status(ctx, rc, "sb_tsne"));
    std::vector<u64> counts, shape;
    SB_TRY(comm_allgather_u64_host(ctx, n_local, counts));
    SB_TRY(comm_allgather_u64_host(ctx, ((u64)k << 32) | dim, shape));
    u64 n = 0, maxr = 0, off = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        if (shape[r] != (((u64)k << 32) | dim)) return sb_fail(SB_ERR_INVALID_ARG, "sb_tsne: k or dim differs between ranks (rank %d)", r);
        if (r < ctx->rank) off += counts[r];
        n += counts[r];
        maxr = std::max(maxr, counts[r]);
    }
    // the checks against the global n (the same on every rank)
    SB_TRY(ts_knn_args(n, dim, k, o.perplexity, "sb_tsne"));
    DevBuf<double> dX, dS, dU, db;
    DevBuf<u32> dn;
    SB_TRY(dX.alloc(n * dim));
    SB_TRY(dn.alloc(n * k));
    SB_TRY(dU.alloc(o.init == SB_TSNE_INIT_USER ? 2 * n : 0));
    if (ctx->nranks == 1) {
        SB_CUDA(cudaMemcpyAsync(dX.p, X, n * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(dn.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        if (o.init == SB_TSNE_INIT_USER) SB_CUDA(cudaMemcpyAsync(dU.p, init, 2 * n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    } else {
        TraceScope tr(ctx, "tsne: row all-gather");
        SB_TRY(um_gather_rows(ctx, X, n_local, 2 * (u64)dim, counts, maxr, (u32 *)dX.p));
        SB_TRY(um_gather_rows(ctx, nbr, n_local, k, counts, maxr, dn.p));
        if (o.init == SB_TSNE_INIT_USER) SB_TRY(um_gather_rows(ctx, init, n_local, 4, counts, maxr, (u32 *)dU.p));
    }
    DevBuf<double> Y;
    if (o.init == SB_TSNE_INIT_USER) SB_TRY(ts_init(ctx, dU.p, n, 2, o, Y, "sb_tsne"));
    else SB_TRY(ts_init(ctx, dX.p, n, dim, o, Y, "sb_tsne"));
    dU.release();
    UmGraph g;
    SB_TRY(ts_affinities(ctx, dX.p, dn.p, n, dim, k, o.perplexity, g, db, "sb_tsne"));
    dX.release();
    dn.release();
    db.release();
    SB_TRY(ts_layout(ctx, g, Y, o, info));
    return ts_copy_out(ctx, Y, off, n_local, out);
}
