// cluster.cu -- graph clustering of the kNN lists: the shared-nearest-neighbour graph and deterministic Louvain (the step between
// kNN and differential expression; the reference's `leiden` crate provides Louvain as the base of its algorithms).  The rules are
// stated beside the entry points in include/scanb200.h and restated, literally, by oracle/louvain.py.
//
//   snn graph   k_snn_rows validates every row and writes its sorted closed neighbourhood N(i) u {i} plus both directed pairs of
//               every listed neighbour; a 64-bit key radix sort + unique gives the symmetric CSR (rows by binary search), and
//               k_snn_weights intersects the two sorted lists of an edge (a thread per edge, lists <= 129 long).
//   moving      per node, the weights to every neighbouring community, by degree: a warp per node with a 256-slot shared table
//               (degree <= 128; lanes holding the same community elect one inserter with __match_any_sync), a CTA per node with
//               a shared table of up to 16,384 slots (degree <= 8,192), and beyond that a global sort + reduce-by-key of just those
//               nodes' (node, community) pairs.  Every sum is an integer, so the path cannot change a result.
//   evaluate    S by u64 atomics, the intra-community weight and the 128-bit sum of S_c^2 by block reductions + atomics; the host
//               reads five words per iteration (the only round trip) and keeps or reverts the moves.
//   aggregate   dense renumbering (flag + scan), coarse edges by a sort of (c_i << 32 | c_j) keys and a reduce-by-key.
// Weights are fixed-point integers (the SNN graph: Jaccard index << 24), so every total is exact and the result is independent of
// the order atomics land in: the device result equals the oracle bit for bit.
#include <cmath>

#include <cub/cub.cuh>

#include "common.cuh"

#define CL_PAD 0xFFFFFFFFu
#define SNN_MAX_K 128
#define SNN_SCALE_BITS 24
#define LV_WARP_DEG 128       // warp path: degree bound and its table (load <= 1/2)
#define LV_WARP_TS 256
#define LV_WARPS 8            // warps (nodes in flight) per block of the warp path
#define LV_CTA_DEG 8192       // CTA path: degree bound; its table is the next power of two >= 2 x the largest degree in the class
#define LV_CTA_THREADS 512
#define LV_MAX_SUM ((u64)1 << 53)

typedef unsigned long long ull;

// ---------------------------------------------------------------- small helpers
static int cl_grid(sb_ctx *ctx, u64 items, int per_block) {
    return (int)std::max<u64>(1, std::min<u64>((items + per_block - 1) / per_block, (u64)ctx->sm_count * 32));
}

__device__ __forceinline__ void add128(ull &hi, ull &lo, ull h2, ull l2) {
    const ull s = lo + l2;
    hi += h2 + (s < lo ? 1ull : 0ull);
    lo = s;
}
// exact 128-bit accumulation: the low word's carry is counted by the thread whose add wrapped it
__device__ __forceinline__ void atomic_add128(ull *acc /* [lo, hi] */, ull hi, ull lo) {
    if (lo) {
        const ull old = atomicAdd(acc, lo);
        if (old + lo < old) hi++;
    }
    if (hi) atomicAdd(acc + 1, hi);
}
// block-wide 128-bit sum of every thread's (hi, lo), one atomic per block (blockDim.x a multiple of 32, <= 1024)
__device__ __forceinline__ void block_add128(ull *acc, ull hi, ull lo) {
    __shared__ ull s_hi[32], s_lo[32];
    for (int o = 16; o > 0; o >>= 1) add128(hi, lo, __shfl_xor_sync(0xffffffffu, hi, o), __shfl_xor_sync(0xffffffffu, lo, o));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) {
        s_hi[warp] = hi;
        s_lo[warp] = lo;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        ull h = 0, l = 0;
        for (int k = 0; k < (int)(blockDim.x >> 5); k++) add128(h, l, s_hi[k], s_lo[k]);
        atomic_add128(acc, h, l);
    }
}

__global__ void k_iota(u32 *a, u64 n) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) a[i] = (u32)i;
}
// first position with keys[pos] >= (r << 32), for every row r in [0, n]
__global__ void k_rows_from_keys(const u64 *__restrict__ keys, u64 nnz, u64 n, u64 *__restrict__ ptr) {
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
__global__ void k_split_keys(const u64 *__restrict__ keys, u64 nnz, u32 *__restrict__ idx) {
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (u64)gridDim.x * blockDim.x) idx[e] = (u32)keys[e];
}

// CUB calls with their temporary storage
static int sort_keys(sb_ctx *ctx, DevBuf<u64> &keys, u64 count) {
    DevBuf<u64> out;
    SB_TRY(out.alloc(count));
    size_t tb = 0;
    SB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb, keys.p, out.p, count, 0, 64, ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tb));
    SB_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, tb, keys.p, out.p, count, 0, 64, ctx->stream));
    count_launch(ctx, false);
    keys.swap(out);
    return SB_OK;
}
int sort_pairs(sb_ctx *ctx, DevBuf<u64> &keys, DevBuf<u64> &vals, u64 count) {
    DevBuf<u64> ko, vo;
    SB_TRY(ko.alloc(count));
    SB_TRY(vo.alloc(count));
    size_t tb = 0;
    SB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb, keys.p, ko.p, vals.p, vo.p, count, 0, 64, ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tb));
    SB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tb, keys.p, ko.p, vals.p, vo.p, count, 0, 64, ctx->stream));
    count_launch(ctx, false);
    keys.swap(ko);
    vals.swap(vo);
    return SB_OK;
}
// equal adjacent keys summed (u64): keys / vals replaced by the runs, *runs their number
static int reduce_by_key(sb_ctx *ctx, DevBuf<u64> &keys, DevBuf<u64> &vals, u64 count, u64 *runs) {
    DevBuf<u64> ko, vo, nr;
    SB_TRY(ko.alloc(count));
    SB_TRY(vo.alloc(count));
    SB_TRY(nr.alloc(1));
    size_t tb = 0;
    SB_CUDA(cub::DeviceReduce::ReduceByKey(nullptr, tb, keys.p, ko.p, vals.p, vo.p, nr.p, cuda::std::plus<u64>{}, count, ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tb));
    SB_CUDA(cub::DeviceReduce::ReduceByKey(tmp.p, tb, keys.p, ko.p, vals.p, vo.p, nr.p, cuda::std::plus<u64>{}, count, ctx->stream));
    count_launch(ctx, false);
    SB_CUDA(cudaMemcpyAsync(runs, nr.p, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    keys.swap(ko);
    vals.swap(vo);
    return SB_OK;
}

// A weighted graph on the device: symmetric CSR, u64 fixed-point weights.
struct DevGraph {
    u64 n = 0, nnz = 0;
    DevBuf<u64> ptr;  // [n + 1]
    DevBuf<u32> idx;  // [nnz]
    DevBuf<u64> w;    // [nnz]
};

// ---------------------------------------------------------------- shared-nearest-neighbour graph
// thread per row: validation (bits: 1 index >= n, 2 self index, 4 duplicate, 8 padding before the row end), the sorted closed
// neighbourhood into cl[i * (k + 1) ..] (length clen[i]), both directed pairs of every listed neighbour (all-ones key: none)
__global__ void k_snn_rows(const u32 *__restrict__ nbr, u64 n, u32 k, u32 *__restrict__ cl, u32 *__restrict__ clen, u64 *__restrict__ keys,
                           int *__restrict__ err) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u32 *r = nbr + i * k;
        u32 *o = cl + i * (k + 1);
        u64 *kk = keys + 2 * i * k;
        u32 len = 0;
        int e = 0;
        bool padded = false;
        for (u32 t = 0; t < k; t++) {
            const u32 j = r[t];
            kk[2 * t] = kk[2 * t + 1] = ~0ull;
            if (j == CL_PAD) {
                padded = true;
                continue;
            }
            if (padded) e |= 8;
            if (j >= n) {
                e |= 1;
                continue;
            }
            if (j == i) {
                e |= 2;
                continue;
            }
            kk[2 * t] = (i << 32) | j;
            kk[2 * t + 1] = ((u64)j << 32) | i;
            o[len++] = j;
        }
        o[len++] = (u32)i;
        for (u32 a = 1; a < len; a++) {  // insertion sort (<= 129 entries)
            const u32 v = o[a];
            u32 b = a;
            while (b > 0 && o[b - 1] > v) {
                o[b] = o[b - 1];
                b--;
            }
            o[b] = v;
        }
        for (u32 a = 1; a < len; a++)
            if (o[a] == o[a - 1]) e |= 4;
        clen[i] = len;
        if (e) atomicOr(err, e);
    }
}

// thread per edge: s = |N+(i) n N+(j)| by merging the sorted lists, w = (s << 24) / (|N+(i)| + |N+(j)| - s)
__global__ void k_snn_weights(const u64 *__restrict__ keys, u64 nnz, u32 k, const u32 *__restrict__ cl, const u32 *__restrict__ clen,
                              u32 *__restrict__ idx, u64 *__restrict__ w) {
    for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (u64)gridDim.x * blockDim.x) {
        const u64 key = keys[e];
        const u32 i = (u32)(key >> 32), j = (u32)key;
        const u32 *a = cl + (u64)i * (k + 1), *b = cl + (u64)j * (k + 1);
        const u32 la = clen[i], lb = clen[j];
        u32 p = 0, q = 0, s = 0;
        while (p < la && q < lb) {
            const u32 x = a[p], y = b[q];
            s += x == y;
            p += x <= y;
            q += y <= x;
        }
        idx[e] = j;
        w[e] = ((u64)s << SNN_SCALE_BITS) / (u64)(la + lb - s);
    }
}

// nbr: device rows [n x k] (global indices) -> g
static int snn_build(sb_ctx *ctx, const u32 *d_nbr, u64 n, u32 k, DevGraph &g) {
    TraceScope tr(ctx, "cluster: snn graph");
    const u64 np = 2 * n * k;
    DevBuf<u32> cl, clen;
    DevBuf<u64> keys;
    DevBuf<int> err;
    SB_TRY(cl.alloc(n * (k + 1)));
    SB_TRY(clen.alloc(n));
    SB_TRY(keys.alloc(np));
    SB_TRY(err.alloc(1));
    SB_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), ctx->stream));
    k_snn_rows<<<cl_grid(ctx, n, 128), 128, 0, ctx->stream>>>(d_nbr, n, k, cl.p, clen.p, keys.p, err.p);
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    int herr = 0;
    SB_CUDA(cudaMemcpyAsync(&herr, err.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (herr)
        return sb_fail(SB_ERR_INVALID_ARG, "sb_snn_graph: invalid neighbour lists:%s%s%s%s", herr & 1 ? " an index >= n" : "", herr & 2 ? " a self index" : "",
                       herr & 4 ? " a duplicate in a row" : "", herr & 8 ? " padding before the row end" : "");
    SB_TRY(sort_keys(ctx, keys, np));
    // unique keys; the all-ones key of unused slots sorts last and is dropped
    DevBuf<u64> uq, nu;
    SB_TRY(uq.alloc(np));
    SB_TRY(nu.alloc(1));
    size_t tb = 0;
    SB_CUDA(cub::DeviceSelect::Unique(nullptr, tb, keys.p, uq.p, nu.p, np, ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tb));
    SB_CUDA(cub::DeviceSelect::Unique(tmp.p, tb, keys.p, uq.p, nu.p, np, ctx->stream));
    count_launch(ctx, false);
    u64 nuniq = 0, last = 0;
    SB_CUDA(cudaMemcpyAsync(&nuniq, nu.p, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (nuniq) {
        SB_CUDA(cudaMemcpyAsync(&last, uq.p + nuniq - 1, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    g.n = n;
    g.nnz = nuniq - (nuniq && last == ~0ull ? 1 : 0);
    SB_TRY(g.ptr.alloc(n + 1));
    SB_TRY(g.idx.alloc(g.nnz));
    SB_TRY(g.w.alloc(g.nnz));
    k_rows_from_keys<<<cl_grid(ctx, n + 1, 256), 256, 0, ctx->stream>>>(uq.p, g.nnz, n, g.ptr.p);
    if (g.nnz) k_snn_weights<<<cl_grid(ctx, g.nnz, 256), 256, 0, ctx->stream>>>(uq.p, g.nnz, k, cl.p, clen.p, g.idx.p, g.w.p);
    count_launch(ctx);
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- Louvain: strengths, evaluation
// warp per node: K[i] = row sum (a self loop counted once); acc[0..1] += K[i] (128-bit)
__global__ void k_lv_strength(const u64 *__restrict__ ptr, const u64 *__restrict__ w, u64 n, u64 *__restrict__ K, ull *__restrict__ acc) {
    const int lane = threadIdx.x & 31;
    ull hi = 0, lo = 0;
    for (u64 i = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += ((u64)gridDim.x * blockDim.x) >> 5) {
        u64 s = 0;
        for (u64 x = ptr[i] + lane; x < ptr[i + 1]; x += 32) s += w[x];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            K[i] = s;
            add128(hi, lo, 0, s);
        }
    }
    block_add128(acc, hi, lo);
}
__global__ void k_lv_tot(const u32 *__restrict__ C, const u64 *__restrict__ K, u64 n, ull *__restrict__ S) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (K[i]) atomicAdd(&S[C[i]], (ull)K[i]);
}
// warp per node: acc[0] += weight of its edges inside its community (self loop included)
__global__ void k_lv_intra(const u64 *__restrict__ ptr, const u32 *__restrict__ idx, const u64 *__restrict__ w, const u32 *__restrict__ C, u64 n,
                           ull *__restrict__ acc) {
    const int lane = threadIdx.x & 31;
    ull hi = 0, lo = 0;
    for (u64 i = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += ((u64)gridDim.x * blockDim.x) >> 5) {
        const u32 c = C[i];
        u64 s = 0;
        for (u64 x = ptr[i] + lane; x < ptr[i + 1]; x += 32) s += C[idx[x]] == c ? w[x] : 0;
        add128(hi, lo, 0, s);
    }
    block_add128(acc, hi, lo);
}
// acc[0..1] += sum_c S_c^2 (exact, 128-bit)
__global__ void k_lv_sq(const u64 *__restrict__ S, u64 n, ull *__restrict__ acc) {
    ull hi = 0, lo = 0;
    for (u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (u64)gridDim.x * blockDim.x) {
        const u64 s = S[c];
        add128(hi, lo, __umul64hi(s, s), s * s);
    }
    block_add128(acc, hi, lo);
}

// ---------------------------------------------------------------- Louvain: local moving
struct MoveArgs {
    const u64 *ptr;
    const u32 *idx;
    const u64 *w;
    const u64 *K;
    const u32 *C;
    const u64 *S;
    u32 *Cn;
    int *moved;
    double g2m;
    int up;
};

// gain(c) = ((double)e_ic - (double)e_ia) - g2m (double)K_i ((double)S_c - (double)(S_a - K_i)), in this order, no contraction
__device__ __forceinline__ double lv_gain(u64 e_ic, double e_ia, double kg, u64 S_c, double s_rest) {
    return __dsub_rn(__dsub_rn((double)e_ic, e_ia), __dmul_rn(kg, __dsub_rn((double)S_c, s_rest)));
}
// (g, c) beats (bg, bc): a larger gain, or the same gain and a smaller community
__device__ __forceinline__ void lv_better(double &bg, u32 &bc, double g, u32 c) {
    if (g > bg || (g == bg && c < bc)) {
        bg = g;
        bc = c;
    }
}

__device__ __forceinline__ u32 tab_insert(u32 *keys, u32 ts, u32 c) {
    u32 h = (c * 2654435761u) & (ts - 1);
    while (true) {
        const u32 prev = atomicCAS(&keys[h], CL_PAD, c);
        if (prev == CL_PAD || prev == c) return h;
        h = (h + 1) & (ts - 1);
    }
}
__device__ __forceinline__ u64 tab_find(const u32 *keys, const ull *vals, u32 ts, u32 c) {
    u32 h = (c * 2654435761u) & (ts - 1);
    while (true) {
        const u32 k = keys[h];
        if (k == c) return vals[h];
        if (k == CL_PAD) return 0;
        h = (h + 1) & (ts - 1);
    }
}

// A group (a warp, or the whole CTA) per node of `nodes`: e_ic of every neighbouring community into an open-addressing table in
// shared memory, then the best allowed move.  CTA = false: LV_WARPS warps per block, table LV_WARP_TS each; CTA = true: one table
// of ts slots.  Cn[i] = the chosen community, or C[i].
template <bool CTA>
__global__ void __launch_bounds__(CTA ? LV_CTA_THREADS : 32 * LV_WARPS) k_lv_move(MoveArgs a, const u32 *__restrict__ nodes, u64 count, u32 ts) {
    extern __shared__ ull lv_smem[];
    __shared__ double red_g[32];
    __shared__ u32 red_c[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u32 gsize = CTA ? blockDim.x : 32, gtid = CTA ? threadIdx.x : lane, gid = CTA ? 0 : warp;
    const u32 per_block = CTA ? 1 : blockDim.x >> 5;
    ull *vals = lv_smem + (u64)gid * ts;
    u32 *keys = (u32 *)(lv_smem + (u64)per_block * ts) + (u64)gid * ts;
    auto gsync = [&]() {
        if (CTA) __syncthreads();
        else __syncwarp();
    };
    for (u32 s = gtid; s < ts; s += gsize) {
        keys[s] = CL_PAD;
        vals[s] = 0;
    }
    gsync();
    for (u64 q = (u64)blockIdx.x * per_block + gid; q < count; q += (u64)gridDim.x * per_block) {
        const u32 i = nodes[q], ca = a.C[i];
        const u64 b = a.ptr[i], e = a.ptr[i + 1];
        for (u64 base = b; base < e; base += gsize) {  // whole chunks: every warp is converged at the match
            const u64 x = base + gtid;
            u32 c = CL_PAD;
            ull wt = 0;
            if (x < e) {
                const u32 j = a.idx[x];
                if (j != i) {
                    c = a.C[j];
                    wt = a.w[x];
                }
            }
            const unsigned peers = __match_any_sync(0xffffffffu, c);
            const int leader = __ffs(peers) - 1;
            u32 slot = 0;
            if (lane == leader && c != CL_PAD) slot = tab_insert(keys, ts, c);
            slot = __shfl_sync(0xffffffffu, slot, leader);
            if (c != CL_PAD) atomicAdd(&vals[slot], wt);
        }
        gsync();
        const u64 Ki = a.K[i];
        const double e_ia = (double)tab_find(keys, vals, ts, ca), kg = __dmul_rn(a.g2m, (double)Ki), s_rest = (double)(a.S[ca] - Ki);
        gsync();
        double bg = 0.0;
        u32 bc = CL_PAD;
        for (u32 s = gtid; s < ts; s += gsize) {
            const u32 c = keys[s];
            if (c == CL_PAD) continue;
            if (a.up ? c > ca : c < ca) {
                const double g = lv_gain(vals[s], e_ia, kg, a.S[c], s_rest);
                if (g > 0.0) lv_better(bg, bc, g, c);
            }
            keys[s] = CL_PAD;
            vals[s] = 0;
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double g2 = __shfl_xor_sync(0xffffffffu, bg, o);
            const u32 c2 = __shfl_xor_sync(0xffffffffu, bc, o);
            lv_better(bg, bc, g2, c2);
        }
        if (CTA) {
            if (lane == 0) {
                red_g[warp] = bg;
                red_c[warp] = bc;
            }
            __syncthreads();
            if (threadIdx.x == 0)
                for (int k = 1; k < (int)(blockDim.x >> 5); k++) lv_better(bg, bc, red_g[k], red_c[k]);
        }
        if (gtid == 0) {
            a.Cn[i] = bc != CL_PAD ? bc : ca;
            if (bc != CL_PAD) atomicOr(a.moved, 1);
        }
        gsync();
    }
}

// Nodes past the CTA table: their (node, community) pairs sorted and summed in global memory.
// block per listed node q: key = q << 32 | C[j] (self loop: all-ones community), value w
__global__ void k_hv_pairs(MoveArgs a, const u32 *__restrict__ nodes, const u64 *__restrict__ off, u64 *__restrict__ keys, u64 *__restrict__ vals) {
    const u64 q = blockIdx.x;
    const u32 i = nodes[q];
    const u64 b = a.ptr[i], e = a.ptr[i + 1], o = off[q];
    for (u64 x = b + threadIdx.x; x < e; x += blockDim.x) {
        const u32 j = a.idx[x];
        keys[o + x - b] = (q << 32) | (j != i ? a.C[j] : CL_PAD);
        vals[o + x - b] = a.w[x];
    }
}
__global__ void k_hv_eia(MoveArgs a, const u32 *__restrict__ nodes, const u64 *__restrict__ keys, const u64 *__restrict__ sums, u64 runs,
                         u64 *__restrict__ eia) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < runs; r += (u64)gridDim.x * blockDim.x) {
        const u64 q = keys[r] >> 32;
        if ((u32)keys[r] == a.C[nodes[q]]) eia[q] = sums[r];
    }
}
// pass 0: the largest positive gain of every node (positive doubles order as their bits); pass 1: the smallest community reaching it
__global__ void k_hv_best(MoveArgs a, const u32 *__restrict__ nodes, const u64 *__restrict__ keys, const u64 *__restrict__ sums, u64 runs,
                          const u64 *__restrict__ eia, int pass, ull *__restrict__ bestg, u32 *__restrict__ bestc) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < runs; r += (u64)gridDim.x * blockDim.x) {
        const u64 q = keys[r] >> 32;
        const u32 c = (u32)keys[r], i = nodes[q], ca = a.C[i];
        if (c == CL_PAD || !(a.up ? c > ca : c < ca)) continue;
        const u64 Ki = a.K[i];
        const double g = lv_gain(sums[r], (double)eia[q], __dmul_rn(a.g2m, (double)Ki), a.S[c], (double)(a.S[ca] - Ki));
        if (!(g > 0.0)) continue;
        const ull bits = (ull)__double_as_longlong(g);
        if (pass == 0) atomicMax(&bestg[q], bits);
        else if (bits == bestg[q]) atomicMin(&bestc[q], c);
    }
}
__global__ void k_hv_final(MoveArgs a, const u32 *__restrict__ nodes, u64 count, const ull *__restrict__ bestg, const u32 *__restrict__ bestc) {
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < count; q += (u64)gridDim.x * blockDim.x) {
        const u32 i = nodes[q];
        a.Cn[i] = bestg[q] ? bestc[q] : a.C[i];
        if (bestg[q]) atomicOr(a.moved, 1);
    }
}

// nodes by degree class: lists[cls * n + pos]; cnt[cls]; cnt[3] = the largest degree of class 1
__global__ void k_lv_classify(const u64 *__restrict__ ptr, u64 n, u32 *__restrict__ lists, ull *__restrict__ cnt) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const u64 d = ptr[i + 1] - ptr[i];
        const int cls = d <= LV_WARP_DEG ? 0 : d <= LV_CTA_DEG ? 1 : 2;
        lists[cls * n + atomicAdd(&cnt[cls], 1ull)] = (u32)i;
        if (cls == 1) atomicMax(&cnt[3], (ull)d);
    }
}
__global__ void k_hv_degrees(const u64 *__restrict__ ptr, const u32 *__restrict__ nodes, u64 count, u64 *__restrict__ deg) {
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < count; q += (u64)gridDim.x * blockDim.x) deg[q] = ptr[nodes[q] + 1] - ptr[nodes[q]];
}

// ---------------------------------------------------------------- Louvain: aggregation
__global__ void k_ag_mark(const u32 *__restrict__ C, u64 n, u64 *__restrict__ flag) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) flag[C[i]] = 1;
}
__global__ void k_ag_labels(u32 *__restrict__ lab, u64 n0, const u32 *__restrict__ C, const u64 *__restrict__ newid) {
    for (u64 v = (u64)blockIdx.x * blockDim.x + threadIdx.x; v < n0; v += (u64)gridDim.x * blockDim.x) lab[v] = (u32)newid[C[lab[v]]];
}
// warp per row: keys = (c_i << 32 | c_j), values w
__global__ void k_ag_keys(const u64 *__restrict__ ptr, const u32 *__restrict__ idx, const u64 *__restrict__ w, const u32 *__restrict__ C,
                          const u64 *__restrict__ newid, u64 n, u64 *__restrict__ keys, u64 *__restrict__ vals) {
    const int lane = threadIdx.x & 31;
    for (u64 i = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += ((u64)gridDim.x * blockDim.x) >> 5) {
        const u64 ci = newid[C[i]] << 32;
        for (u64 x = ptr[i] + lane; x < ptr[i + 1]; x += 32) {
            keys[x] = ci | newid[C[idx[x]]];
            vals[x] = w[x];
        }
    }
}

// ---------------------------------------------------------------- Louvain: host driver
// S = community totals of C; host[0..1] intra weight, host[2..3] sum S_c^2 (128-bit each), host[4] the moved flag
static int lv_evaluate(sb_ctx *ctx, const DevGraph &g, const u64 *K, const u32 *C, ull *S, ull *acc, ull host[5]) {
    const u64 n = g.n;
    SB_CUDA(cudaMemsetAsync(S, 0, n * sizeof(ull), ctx->stream));
    SB_CUDA(cudaMemsetAsync(acc, 0, 4 * sizeof(ull), ctx->stream));
    k_lv_tot<<<cl_grid(ctx, n, 256), 256, 0, ctx->stream>>>(C, K, n, S);
    k_lv_intra<<<cl_grid(ctx, n * 32, 256), 256, 0, ctx->stream>>>(g.ptr.p, g.idx.p, g.w.p, C, n, acc);
    k_lv_sq<<<cl_grid(ctx, n, 256), 256, 0, ctx->stream>>>((const u64 *)S, n, acc + 2);
    for (int k = 0; k < 3; k++) count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaMemcpyAsync(host, acc, 5 * sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

static double lv_quality(ull intra, ull sq_lo, ull sq_hi, double two_m, double gamma) {
    const double s2 = (double)sq_hi * 18446744073709551616.0 + (double)sq_lo;
    return (double)intra / two_m - (gamma * s2) / (two_m * two_m);
}

struct LvOpts {
    double gamma;
    u32 max_levels, max_iterations;
};

// Louvain on g (consumed: replaced level by level by the coarse graphs) -> labels[n] (by size), info
static int louvain_dev(sb_ctx *ctx, DevGraph &g, const LvOpts &opt, uint32_t *labels, sb_louvain_info *info) {
    memset(info, 0, sizeof(*info));
    const u64 n0 = g.n;
    if (n0 == 0) return SB_OK;
    DevBuf<u32> lab;
    DevBuf<ull> acc;  // [0..1] 128-bit sums, [2..3] 128-bit sums, [4] moved flag
    SB_TRY(lab.alloc(n0));
    SB_TRY(acc.alloc(8));
    k_iota<<<cl_grid(ctx, n0, 256), 256, 0, ctx->stream>>>(lab.p, n0);
    count_launch(ctx);
    double Qfinal = 0.0;
    for (u32 level = 0; level < opt.max_levels; level++) {
        TraceScope tr(ctx, "cluster: louvain level");
        const u64 n = g.n;
        DevBuf<u64> K;
        DevBuf<ull> S, Sn, cnt;
        DevBuf<u32> C, Cn, lists;
        SB_TRY(K.alloc(n));
        SB_TRY(S.alloc(n));
        SB_TRY(Sn.alloc(n));
        SB_TRY(C.alloc(n));
        SB_TRY(Cn.alloc(n));
        SB_TRY(lists.alloc(3 * n));
        SB_TRY(cnt.alloc(4));
        SB_CUDA(cudaMemsetAsync(acc.p, 0, 8 * sizeof(ull), ctx->stream));
        SB_CUDA(cudaMemsetAsync(cnt.p, 0, 4 * sizeof(ull), ctx->stream));
        k_lv_strength<<<cl_grid(ctx, n * 32, 256), 256, 0, ctx->stream>>>(g.ptr.p, g.w.p, n, K.p, acc.p);
        k_lv_classify<<<cl_grid(ctx, n, 256), 256, 0, ctx->stream>>>(g.ptr.p, n, lists.p, cnt.p);
        k_iota<<<cl_grid(ctx, n, 256), 256, 0, ctx->stream>>>(C.p, n);
        for (int k = 0; k < 3; k++) count_launch(ctx);
        ull hs[2], hc[4];
        SB_CUDA(cudaMemcpyAsync(hs, acc.p, 2 * sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(hc, cnt.p, 4 * sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        const u64 two_m_i = hs[0];
        info->level_nodes[level] = n;
        info->n_levels = level + 1;
        if (two_m_i == 0) {  // no edge weight: every node stays its own cluster
            info->level_iterations[level] = 0;
            info->level_modularity[level] = 0.0;
            break;
        }
        const double two_m = (double)two_m_i, g2m = opt.gamma / two_m;
        // the nodes past the CTA table: their pair offsets
        const u64 n_warp = hc[0], n_cta = hc[1], n_hv = hc[2];
        u32 cta_ts = 2;
        while (cta_ts < 2 * hc[3]) cta_ts <<= 1;
        std::vector<u64> hv_off(n_hv + 1, 0);
        DevBuf<u64> d_off;
        SB_TRY(d_off.alloc(n_hv + 1));
        if (n_hv) {
            DevBuf<u64> deg;
            SB_TRY(deg.alloc(n_hv));
            k_hv_degrees<<<cl_grid(ctx, n_hv, 256), 256, 0, ctx->stream>>>(g.ptr.p, lists.p + 2 * n, n_hv, deg.p);
            count_launch(ctx);
            SB_CUDA(cudaMemcpyAsync(hv_off.data() + 1, deg.p, n_hv * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
            SB_CUDA(cudaStreamSynchronize(ctx->stream));
            for (u64 q = 0; q < n_hv; q++) hv_off[q + 1] += hv_off[q];
            SB_CUDA(cudaMemcpyAsync(d_off.p, hv_off.data(), (n_hv + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        }
        ull h[5];
        SB_TRY(lv_evaluate(ctx, g, K.p, C.p, S.p, acc.p, h));
        double Q = lv_quality(h[0], h[2], h[3], two_m, opt.gamma);
        const size_t warp_smem = (size_t)LV_WARPS * LV_WARP_TS * (sizeof(ull) + sizeof(u32));
        const size_t cta_smem = (size_t)cta_ts * (sizeof(ull) + sizeof(u32));
        if (n_cta) SB_CUDA(cudaFuncSetAttribute(k_lv_move<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cta_smem));
        u32 fails = 0, it = 0;
        bool accepted = false;
        for (u32 t = 0; t < opt.max_iterations; t++) {
            it = t + 1;
            SB_CUDA(cudaMemsetAsync(acc.p + 4, 0, sizeof(ull), ctx->stream));
            MoveArgs a{g.ptr.p, g.idx.p, g.w.p, K.p, C.p, (const u64 *)S.p, Cn.p, (int *)(acc.p + 4), g2m, (int)(t % 2 == 0)};
            if (n_warp) {
                const u64 blocks = std::min<u64>((n_warp + LV_WARPS - 1) / LV_WARPS, (u64)ctx->sm_count * 16);
                k_lv_move<false><<<(unsigned)blocks, 32 * LV_WARPS, warp_smem, ctx->stream>>>(a, lists.p, n_warp, LV_WARP_TS);
                count_launch(ctx);
            }
            if (n_cta) {
                k_lv_move<true><<<(unsigned)std::min<u64>(n_cta, (u64)ctx->sm_count * 2), LV_CTA_THREADS, cta_smem, ctx->stream>>>(a, lists.p + n, n_cta, cta_ts);
                count_launch(ctx);
            }
            if (n_hv) {
                const u64 np = hv_off[n_hv];
                DevBuf<u64> keys, vals, eia;
                DevBuf<ull> bestg;
                DevBuf<u32> bestc;
                SB_TRY(keys.alloc(np));
                SB_TRY(vals.alloc(np));
                SB_TRY(eia.alloc(n_hv));
                SB_TRY(bestg.alloc(n_hv));
                SB_TRY(bestc.alloc(n_hv));
                k_hv_pairs<<<(unsigned)n_hv, 256, 0, ctx->stream>>>(a, lists.p + 2 * n, d_off.p, keys.p, vals.p);
                count_launch(ctx);
                SB_TRY(sort_pairs(ctx, keys, vals, np));
                u64 runs = 0;
                SB_TRY(reduce_by_key(ctx, keys, vals, np, &runs));
                SB_CUDA(cudaMemsetAsync(eia.p, 0, n_hv * sizeof(u64), ctx->stream));
                SB_CUDA(cudaMemsetAsync(bestg.p, 0, n_hv * sizeof(ull), ctx->stream));
                SB_CUDA(cudaMemsetAsync(bestc.p, 0xFF, n_hv * sizeof(u32), ctx->stream));
                const u32 *hl = lists.p + 2 * n;
                k_hv_eia<<<cl_grid(ctx, runs, 256), 256, 0, ctx->stream>>>(a, hl, keys.p, vals.p, runs, eia.p);
                k_hv_best<<<cl_grid(ctx, runs, 256), 256, 0, ctx->stream>>>(a, hl, keys.p, vals.p, runs, eia.p, 0, bestg.p, bestc.p);
                k_hv_best<<<cl_grid(ctx, runs, 256), 256, 0, ctx->stream>>>(a, hl, keys.p, vals.p, runs, eia.p, 1, bestg.p, bestc.p);
                k_hv_final<<<cl_grid(ctx, n_hv, 256), 256, 0, ctx->stream>>>(a, hl, n_hv, bestg.p, bestc.p);
                for (int k = 0; k < 4; k++) count_launch(ctx);
            }
            SB_CUDA(cudaGetLastError());
            SB_TRY(lv_evaluate(ctx, g, K.p, Cn.p, Sn.p, acc.p, h));
            if (h[4]) {
                const double Qn = lv_quality(h[0], h[2], h[3], two_m, opt.gamma);
                if (Qn > Q) {
                    C.swap(Cn);
                    S.swap(Sn);
                    Q = Qn;
                    fails = 0;
                    accepted = true;
                    continue;
                }
            }
            if (++fails >= 2) break;
        }
        info->level_iterations[level] = it;
        info->level_modularity[level] = Q;
        Qfinal = Q;
        if (!accepted) break;
        // aggregation: communities numbered densely in ascending id, coarse edges summed per (c_i, c_j)
        TraceScope tra(ctx, "cluster: aggregation");
        DevBuf<u64> newid;
        SB_TRY(newid.alloc(n + 1));
        SB_CUDA(cudaMemsetAsync(newid.p, 0, (n + 1) * sizeof(u64), ctx->stream));
        k_ag_mark<<<cl_grid(ctx, n, 256), 256, 0, ctx->stream>>>(C.p, n, newid.p);
        count_launch(ctx);
        {
            DevBuf<u64> sc;
            SB_TRY(sc.alloc(n + 1));
            size_t tb = 0;
            SB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tb, newid.p, sc.p, n + 1, ctx->stream));
            DevBuf<char> tmp;
            SB_TRY(tmp.alloc(tb));
            SB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, newid.p, sc.p, n + 1, ctx->stream));
            count_launch(ctx, false);
            newid.swap(sc);
        }
        u64 nc = 0;
        SB_CUDA(cudaMemcpyAsync(&nc, newid.p + n, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        k_ag_labels<<<cl_grid(ctx, n0, 256), 256, 0, ctx->stream>>>(lab.p, n0, C.p, newid.p);
        DevBuf<u64> keys, vals;
        SB_TRY(keys.alloc(g.nnz));
        SB_TRY(vals.alloc(g.nnz));
        k_ag_keys<<<cl_grid(ctx, n * 32, 256), 256, 0, ctx->stream>>>(g.ptr.p, g.idx.p, g.w.p, C.p, newid.p, n, keys.p, vals.p);
        count_launch(ctx);
        count_launch(ctx);
        SB_TRY(sort_pairs(ctx, keys, vals, g.nnz));
        u64 runs = 0;
        SB_TRY(reduce_by_key(ctx, keys, vals, g.nnz, &runs));
        DevGraph cg;
        cg.n = nc;
        cg.nnz = runs;
        SB_TRY(cg.ptr.alloc(nc + 1));
        SB_TRY(cg.idx.alloc(runs));
        k_rows_from_keys<<<cl_grid(ctx, nc + 1, 256), 256, 0, ctx->stream>>>(keys.p, runs, nc, cg.ptr.p);
        k_split_keys<<<cl_grid(ctx, runs, 256), 256, 0, ctx->stream>>>(keys.p, runs, cg.idx.p);
        count_launch(ctx);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
        cg.w.swap(vals);
        g.n = cg.n;
        g.nnz = cg.nnz;
        g.ptr.swap(cg.ptr);
        g.idx.swap(cg.idx);
        g.w.swap(cg.w);
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    // compose: lab holds the final community of every node; renumber by size, descending, ties to the smallest member
    std::vector<u32> hl(n0);
    SB_CUDA(cudaMemcpyAsync(hl.data(), lab.p, n0 * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    std::vector<u64> size(n0, 0), first(n0, ~0ull);
    for (u64 v = 0; v < n0; v++) {
        size[hl[v]]++;
        if (first[hl[v]] == ~0ull) first[hl[v]] = v;
    }
    std::vector<u32> ids;
    for (u64 c = 0; c < n0; c++)
        if (size[c]) ids.push_back((u32)c);
    std::sort(ids.begin(), ids.end(), [&](u32 x, u32 y) { return size[x] != size[y] ? size[x] > size[y] : first[x] < first[y]; });
    std::vector<u32> rank(n0, 0);
    for (size_t r = 0; r < ids.size(); r++) rank[ids[r]] = (u32)r;
    for (u64 v = 0; v < n0; v++) labels[v] = rank[hl[v]];
    info->n_clusters = (u32)ids.size();
    info->modularity = Qfinal;
    return SB_OK;
}

static int lv_opts(const sb_louvain_opts *o, LvOpts &out, const char *fn) {
    out = LvOpts{1.0, SB_LOUVAIN_MAX_LEVELS, 100};
    if (!o) return SB_OK;
    if (!(o->resolution > 0.0) || !std::isfinite(o->resolution)) return sb_fail(SB_ERR_INVALID_ARG, "%s: resolution must be finite and > 0", fn);
    if (o->max_levels < 1 || o->max_levels > SB_LOUVAIN_MAX_LEVELS)
        return sb_fail(SB_ERR_INVALID_ARG, "%s: max_levels must be 1..%d", fn, SB_LOUVAIN_MAX_LEVELS);
    if (o->max_iterations < 1) return sb_fail(SB_ERR_INVALID_ARG, "%s: max_iterations must be >= 1", fn);
    out = LvOpts{o->resolution, o->max_levels, o->max_iterations};
    return SB_OK;
}

static int snn_args(const uint32_t *nbr, uint64_t n, uint32_t k, const char *fn) {
    if (n && !nbr) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn);
    if (k == 0) return sb_fail(SB_ERR_INVALID_ARG, "%s: k must be >= 1", fn);
    if (k > SNN_MAX_K) return sb_fail(SB_ERR_UNSUPPORTED, "%s: k must be <= %d", fn, SNN_MAX_K);
    if (n >= 0xFFFFFFFFull || n * k >= ((u64)1 << 28))
        return sb_fail(SB_ERR_UNSUPPORTED, "%s: n x k must be below 2^28 (the weight total 2m must stay below 2^53)", fn);
    return SB_OK;
}

// ---------------------------------------------------------------- entry points
extern "C" int sb_snn_graph(sb_ctx *ctx, const uint32_t *nbr, uint64_t n, uint32_t k, uint64_t *indptr, uint32_t *indices, uint64_t *weights,
                            uint64_t *nnz) {
    if (!ctx || !indptr || !nnz || (n && k && (!indices || !weights))) return sb_fail(SB_ERR_INVALID_ARG, "sb_snn_graph: NULL argument");
    SB_TRY(snn_args(nbr, n, k, "sb_snn_graph"));
    SB_ENTER(ctx);
    DevBuf<u32> d_nbr;
    SB_TRY(d_nbr.alloc(n * k));
    if (n) SB_CUDA(cudaMemcpyAsync(d_nbr.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    DevGraph g;
    SB_TRY(snn_build(ctx, d_nbr.p, n, k, g));
    SB_CUDA(cudaMemcpyAsync(indptr, g.ptr.p, (n + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    if (g.nnz) {
        SB_CUDA(cudaMemcpyAsync(indices, g.idx.p, g.nnz * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(weights, g.w.p, g.nnz * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    *nnz = g.nnz;
    return SB_OK;
}

// thread per entry of the row-sorted copy: bits 1 index >= n, 2 asymmetric (pair or weight), 4 duplicate entry
__global__ void k_lv_check(const u64 *__restrict__ fk, const u64 *__restrict__ fv, const u64 *__restrict__ tk, const u64 *__restrict__ tv, u64 nnz, u64 n,
                           int *__restrict__ err) {
    for (u64 x = (u64)blockIdx.x * blockDim.x + threadIdx.x; x < nnz; x += (u64)gridDim.x * blockDim.x) {
        int e = 0;
        if ((u32)fk[x] >= n) e |= 1;
        if (fk[x] != tk[x] || fv[x] != tv[x]) e |= 2;
        if (x && fk[x] == fk[x - 1]) e |= 4;
        if (e) atomicOr(err, e);
    }
}
// warp per row: forward keys (i << 32 | j) and transposed keys (j << 32 | i), both with the weight; acc += w (128-bit)
__global__ void k_lv_pairs(const u64 *__restrict__ ptr, const u32 *__restrict__ idx, const u64 *__restrict__ w, u64 n, u64 *__restrict__ fk,
                           u64 *__restrict__ fv, u64 *__restrict__ tk, u64 *__restrict__ tv, ull *__restrict__ acc) {
    const int lane = threadIdx.x & 31;
    ull hi = 0, lo = 0;
    for (u64 i = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += ((u64)gridDim.x * blockDim.x) >> 5)
        for (u64 x = ptr[i] + lane; x < ptr[i + 1]; x += 32) {
            const u64 j = idx[x];
            fk[x] = (i << 32) | j;
            tk[x] = (j << 32) | i;
            fv[x] = tv[x] = w[x];
            add128(hi, lo, 0, w[x]);
        }
    block_add128(acc, hi, lo);
}

extern "C" int sb_louvain(sb_ctx *ctx, uint64_t n, const uint64_t *indptr, const uint32_t *indices, const uint64_t *weights, const sb_louvain_opts *opts,
                          uint32_t *labels, sb_louvain_info *info) {
    if (!ctx || !indptr || !info || (n && !labels)) return sb_fail(SB_ERR_INVALID_ARG, "sb_louvain: NULL argument");
    LvOpts o;
    SB_TRY(lv_opts(opts, o, "sb_louvain"));
    if (n >= 0xFFFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "sb_louvain: more than 2^32 - 2 nodes");
    if (indptr[0] != 0) return sb_fail(SB_ERR_INVALID_ARG, "sb_louvain: indptr must start at 0");
    for (u64 i = 0; i < n; i++)
        if (indptr[i + 1] < indptr[i]) return sb_fail(SB_ERR_INVALID_ARG, "sb_louvain: indptr decreases at row %llu", (unsigned long long)i);
    const u64 nnz = indptr[n];
    if (nnz && (!indices || !weights)) return sb_fail(SB_ERR_INVALID_ARG, "sb_louvain: NULL argument");
    SB_ENTER(ctx);
    DevGraph g;
    g.n = n;
    g.nnz = nnz;
    SB_TRY(g.ptr.alloc(n + 1));
    SB_TRY(g.idx.alloc(nnz));
    SB_TRY(g.w.alloc(nnz));
    SB_CUDA(cudaMemcpyAsync(g.ptr.p, indptr, (n + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    if (nnz) {
        SB_CUDA(cudaMemcpyAsync(g.idx.p, indices, nnz * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(g.w.p, weights, nnz * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        // validation: the row-sorted pairs must equal the sorted transposed pairs, weights included, with no repeated pair
        TraceScope tr(ctx, "cluster: csr validation");
        DevBuf<u64> fk, fv, tk, tv;
        DevBuf<ull> acc;
        DevBuf<int> err;
        SB_TRY(fk.alloc(nnz));
        SB_TRY(fv.alloc(nnz));
        SB_TRY(tk.alloc(nnz));
        SB_TRY(tv.alloc(nnz));
        SB_TRY(acc.alloc(2));
        SB_TRY(err.alloc(1));
        SB_CUDA(cudaMemsetAsync(acc.p, 0, 2 * sizeof(ull), ctx->stream));
        SB_CUDA(cudaMemsetAsync(err.p, 0, sizeof(int), ctx->stream));
        k_lv_pairs<<<cl_grid(ctx, n * 32, 256), 256, 0, ctx->stream>>>(g.ptr.p, g.idx.p, g.w.p, n, fk.p, fv.p, tk.p, tv.p, acc.p);
        count_launch(ctx);
        SB_TRY(sort_pairs(ctx, fk, fv, nnz));
        SB_TRY(sort_pairs(ctx, tk, tv, nnz));
        k_lv_check<<<cl_grid(ctx, nnz, 256), 256, 0, ctx->stream>>>(fk.p, fv.p, tk.p, tv.p, nnz, n, err.p);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
        int herr = 0;
        ull tot[2];
        SB_CUDA(cudaMemcpyAsync(&herr, err.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(tot, acc.p, 2 * sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        if (herr & 1) return sb_fail(SB_ERR_INVALID_ARG, "sb_louvain: a column index >= n");
        if (herr & 4) return sb_fail(SB_ERR_INVALID_ARG, "sb_louvain: a duplicate entry");
        if (herr & 2) return sb_fail(SB_ERR_INVALID_ARG, "sb_louvain: the CSR is not symmetric (pairs or weights)");
        if (tot[1] || tot[0] >= LV_MAX_SUM) return sb_fail(SB_ERR_UNSUPPORTED, "sb_louvain: the weight total 2m must be below 2^53");
        // the level-0 graph: columns ascending
        k_split_keys<<<cl_grid(ctx, nnz, 256), 256, 0, ctx->stream>>>(fk.p, nnz, g.idx.p);
        count_launch(ctx);
        g.w.swap(fv);
    }
    return louvain_dev(ctx, g, o, labels, info);
}

extern "C" int sb_cluster_knn(sb_ctx *ctx, const uint32_t *nbr, uint64_t n_local, uint32_t k, const sb_louvain_opts *opts, uint32_t *labels,
                              sb_louvain_info *info) {
    if (!ctx) return sb_fail(SB_ERR_INVALID_ARG, "sb_cluster_knn: NULL argument");
    LvOpts o;
    int rc = (!info || (n_local && !labels)) ? sb_fail(SB_ERR_INVALID_ARG, "sb_cluster_knn: NULL argument") : SB_OK;
    if (rc == SB_OK) rc = lv_opts(opts, o, "sb_cluster_knn");
    if (rc == SB_OK) rc = snn_args(nbr, n_local, k, "sb_cluster_knn");
    SB_ENTER(ctx);
    SB_TRY(agree_status(ctx, rc, "sb_cluster_knn"));
    // the rows of all ranks in global cell order (zero-padded all-gather to the largest shard)
    std::vector<u64> counts, ks;
    SB_TRY(comm_allgather_u64_host(ctx, n_local, counts));
    SB_TRY(comm_allgather_u64_host(ctx, k, ks));
    u64 n = 0, maxr = 0, off = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        if (ks[r] != k) return sb_fail(SB_ERR_INVALID_ARG, "sb_cluster_knn: k differs between ranks (%llu on rank %d)", (unsigned long long)ks[r], r);
        if (r < ctx->rank) off += counts[r];
        n += counts[r];
        maxr = std::max(maxr, counts[r]);
    }
    if (n >= 0xFFFFFFFFull || n * k >= ((u64)1 << 28))
        return sb_fail(SB_ERR_UNSUPPORTED, "sb_cluster_knn: n x k must be below 2^28 over all ranks (the weight total 2m must stay below 2^53)");
    DevBuf<u32> d_nbr;
    SB_TRY(d_nbr.alloc(n * k));
    if (ctx->nranks == 1) {
        if (n) SB_CUDA(cudaMemcpyAsync(d_nbr.p, nbr, n * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    } else {
        TraceScope tr(ctx, "cluster: row all-gather");
        const u64 slab = maxr * k;
        DevBuf<u32> mine, all;
        SB_TRY(mine.alloc(slab));
        SB_TRY(all.alloc(slab * ctx->nranks));
        SB_CUDA(cudaMemsetAsync(mine.p, 0, std::max<u64>(1, slab) * sizeof(u32), ctx->stream));
        if (n_local) SB_CUDA(cudaMemcpyAsync(mine.p, nbr, n_local * k * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        if (slab) {
            ProfScope ps(ctx, PH_COMM);
            SB_NCCL(ncclAllGather(mine.p, all.p, slab, ncclUint32, ctx->comm, ctx->stream));
            count_launch(ctx, false);
        }
        u64 at = 0;
        for (int r = 0; r < ctx->nranks; r++) {
            if (counts[r]) SB_CUDA(cudaMemcpyAsync(d_nbr.p + at * k, all.p + (u64)r * slab, counts[r] * k * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));
            at += counts[r];
        }
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    DevGraph g;
    SB_TRY(snn_build(ctx, d_nbr.p, n, k, g));
    d_nbr.release();
    std::vector<u32> all_labels(n);
    SB_TRY(louvain_dev(ctx, g, o, all_labels.data(), info));
    std::copy(all_labels.begin() + off, all_labels.begin() + off + n_local, labels);
    return SB_OK;
}
