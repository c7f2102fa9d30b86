// planes.cu -- the dense half of the hybrid SpMM on the INTEGER tensor cores (tcgen05.mma kind::i8, accumulators in TMEM).
//
// Where the count matrix is dense enough, a sparse f64 gather (160 B of operand per 8-byte entry, DESIGN.md 3) is the wrong
// tool.  Counts are small integers, so for each count level k = 1..L the indicator [v_gc == k] is a 0/1 matrix M_k, and
//     A^T.Y  :  T[c,:] += sum_k L_c(k) * ( M_k^T-slice . Ys )[c,:]          Ys = row_scale * Y      (restates the products of
//     A.X    :  P[g,:] += sum_k ( M_k . (L_c(k) X) )[g,:]                                           low_rank_offset.rs:68-96)
// with L_c(k) = log_b(col_scale_c * k + 1) the only cell-dependent factor (map.cuh).  The dense f64 operand is cut per column
// into 7 balanced base-256 digits of a 54-bit fixed-point number (Ozaki splitting): every M_k . digit-plane product is an
// EXACT int8 x int8 -> int32 tensor-core product, and the digits are recombined in the epilogue (two int64 halves -> f64,
// one rounding).  The error is that of one rounding to 54 bits of the column maximum per operand entry -- measured against
// the oracle at the same level as the f64 DMMA panel it replaces (tests/test_gpu_parity.py).
//
// Layout ("bit planes"): genes are ranked by how many cells express them; level k keeps the first G_k ranks (multiples of
// 128, G_1 >= G_2 >= ...), chosen so that a (gene, level) pair lives here only if at least `plane_min_density` of the cells
// have exactly that count.  plane_k is bit-packed and tile-transposed: word (tile, gw, cell) = 32 genes [32 gw, 32 gw + 32) of
// cell 128 tile + cell, stored at ((tile * G_k/32) + gw) * 128 + cell -- both products read 128-cell x 32-gene blocks as
// 512 contiguous bytes.  Every entry not covered by a plane stays in the sparse streams (gather.cu).
//
// Kernels (one CTA per SM, warp-specialised: warps 0-3 epilogue, warp 4 MMA issue, warps 5-12 producers):
//   k_planes_t : a CTA keeps the digit planes of 1,024 ranks resident in shared memory as the B operand (K-major, 144 KB),
//                walks cell tiles; producers expand plane words into 0/1 int8 A tiles (K-major core matrices) through an
//                8-stage mbarrier ring; up to three levels accumulate into three TMEM accumulators (3 x 144 columns).
//   k_planes_n : a CTA owns 384 ranks (three 128-gene accumulators) and a range of cell tiles; per 32-cell K step and level
//                the producers expand the plane words into an MN-major A tile and copy the digit rows of L_c(k).X[c,:]
//                (written once per product by k_pl_digits_n) as the MN-major B tile; all levels share the accumulators.
#include <numeric>

#include "common.cuh"
#include "map.cuh"
#include "tc05.cuh"

using namespace tc05;

#define PL_TILE 128u
#define PL_COLS 20u
#define PL_DIG 7u
#define PL_NCOL 144u  // 7 x 20 = 140 digit columns, padded to a multiple of 16 (UMMA N for M = 128)
#define PL_FIX 54
#define PL_NONE 0xFFFFFFFFu

#define PT_RANGE 1024u                          // ranks per resident B block (T side)
#define PT_B_BYTES (PT_RANGE * PL_NCOL)         // 147,456
#define PT_KCHUNK_BYTES (PL_NCOL / 8 * 128)     // 2,304: one 16-gene K chunk of B (18 core matrices)
#define PT_WORDS 2u                             // 32-gene words per sub-stage (a sub-stage feeds PT_WORDS MMAs)
#define PT_STAGE_BYTES (PL_TILE * 32u * PT_WORDS)  // 8,192: a sub-stage = 128 cells x 64 genes of one level
#define PT_NSTAGES 8u                           // sub-stages in the ring, one per producer warp
#define PT_SUB 2u                               // sub-stages per MMA stage: 128 genes, four MMAs per barrier round trip
#define PT_NSTG (PT_NSTAGES / PT_SUB)
#define PT_PROD_WARPS PT_NSTAGES
#define PL_EPI_WARPS 4u
#define PL_PROD_WARPS 8u
#define PL_THREADS ((PL_EPI_WARPS + 1 + PL_PROD_WARPS) * 32)  // 416

#define PN_GROUP 384u                           // ranks per CTA (N side): three M tiles
#define PN_A_BYTES (3u * 4096u)
#define PN_B_BYTES (32u * PL_NCOL)              // 4,608
#define PN_STAGE_BYTES (PN_A_BYTES + PN_B_BYTES)  // 16,896
#define PN_NSTAGES 12u                          // sub-stages (32 cells of one level) in the ring
#define PN_SUB 4u                               // sub-stages per MMA stage: a whole 128-cell tile of one level, up to 12 MMAs
#define PN_NSTG (PN_NSTAGES / PN_SUB)
#define PN_CELLGRP_BYTES (PL_NCOL / 16 * 128)   // 1,152: digit rows of 8 cells (9 core matrices)

struct PlDev {
    u32 *bits[PL_MAX_LEVELS];
    u32 G[PL_MAX_LEVELS];
    u32 L;
    u64 ntiles;
    u64 n;
};

static PlDev make_pldev(const sb_mat *mt) {
    PlDev d;
    memset(&d, 0, sizeof(d));
    d.L = mt->pl.L;
    d.ntiles = mt->pl.ntiles;
    d.n = mt->n;
    for (u32 k = 0; k < mt->pl.L; k++) {
        d.bits[k] = mt->pl.bits[k].p;
        d.G[k] = mt->pl.G[k];
    }
    return d;
}

// ---------------------------------------------------------------- selection of the planes
// hist[k * m + g] += 1 for every entry of the sampled cells with count k + 1 <= L
__global__ void k_pl_level_hist(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, u32 m, u32 L, unsigned long long *__restrict__ hist) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        const u64 s = ptr[c], e = ptr[c + 1];
        for (u64 k = s + lane; k < e; k += 32) {
            const uint2 z = cm[k];
            if (z.y >= 1 && z.y <= L) atomicAdd(&hist[(size_t)(z.y - 1) * m + z.x], 1ull);
        }
    }
}

static void units_round(std::vector<u32> &nctas, const std::vector<double> &cost, u32 total) {
    // largest-remainder apportionment with at least one CTA per unit
    const size_t U = cost.size();
    nctas.assign(U, 1);
    if (U == 0) return;
    double sum = 0.0;
    for (double c : cost) sum += c;
    if (U >= total || sum <= 0.0) return;
    std::vector<double> ideal(U);
    u32 used = 0;
    for (size_t i = 0; i < U; i++) {
        ideal[i] = cost[i] / sum * total;
        nctas[i] = std::max<u32>(1, (u32)ideal[i]);
        used += nctas[i];
    }
    while (used > total) {  // ones forced up to 1 may overshoot: take from the most over-served
        size_t best = 0;
        double worst = -1e300;
        for (size_t i = 0; i < U; i++)
            if (nctas[i] > 1 && (double)nctas[i] - ideal[i] > worst) { worst = (double)nctas[i] - ideal[i]; best = i; }
        nctas[best]--;
        used--;
    }
    while (used < total) {
        size_t best = 0;
        double worst = -1e300;
        for (size_t i = 0; i < U; i++)
            if (ideal[i] - (double)nctas[i] > worst) { worst = ideal[i] - (double)nctas[i]; best = i; }
        nctas[best]++;
        used++;
    }
}

// Chooses the planes from the entry counts of local cells [c0, c1) (the whole shard or the first upload chunk), summed
// over ranks.  Allocates and zeroes the planes, fills hot_idx (rank -> gene), hot_of_gene (gene -> rank) and the unit tables.
int planes_select(sb_mat *mt, u64 c0, u64 c1) {
    sb_ctx *ctx = mt->ctx;
    PlaneSet &pl = mt->pl;
    pl.active = false;
    pl.L = 0;
    const u32 m = mt->m;
    const u32 Lmax = (u32)std::min<int>(std::max(ctx->plane_levels, 1), PL_MAX_LEVELS);
    if (m < 128 || mt->n_global == 0 || ctx->plane_cap < 128) return SB_OK;
    SyncScope tr(ctx, "build: plane selection");
    DevBuf<u64> d_hist;
    const size_t hn = (size_t)Lmax * m + 1;
    SB_TRY(d_hist.alloc(hn));
    SB_CUDA(cudaMemsetAsync(d_hist.p, 0, hn * sizeof(u64), ctx->stream));
    if (c1 > c0) {
        ProfScope ps(ctx, PH_REDUCE);
        u64 blocks = std::min<u64>(((c1 - c0) * 32 + 255) / 256, (u64)ctx->sm_count * 16);
        k_pl_level_hist<<<(unsigned)std::max<u64>(1, blocks), 256, 0, ctx->stream>>>(mt->cm_ptr.p + c0, mt->cm.p, c1 - c0, m, Lmax,
                                                                                     (unsigned long long *)d_hist.p);
        count_launch(ctx);
    }
    const u64 sample = c1 - c0;
    SB_CUDA(cudaMemcpyAsync(d_hist.p + (hn - 1), &sample, sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    SB_TRY(comm_allreduce_u64(ctx, d_hist.p, hn));
    std::vector<u64> h(hn);
    SB_CUDA(cudaMemcpyAsync(h.data(), d_hist.p, hn * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    const double cells = (double)h[hn - 1];
    if (cells <= 0.0) return SB_OK;
    // rank by the number of entries with a count of 1..Lmax (ties: lower gene index)
    std::vector<u64> tot(m, 0);
    for (u32 k = 0; k < Lmax; k++)
        for (u32 g = 0; g < m; g++) tot[g] += h[(size_t)k * m + g];
    std::vector<u32> order(m);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](u32 a, u32 b) { return tot[a] > tot[b]; });
    const u32 cap = std::min<u32>((u32)ctx->plane_cap, m) & ~127u;
    const double thr = ctx->plane_min_density * cells;
    u32 prev = cap;
    u32 L = 0;
    for (u32 k = 0; k < Lmax; k++) {
        u32 G = 0;
        for (u32 b0 = 0; b0 + 128 <= prev; b0 += 128) {  // leading 128-rank blocks whose mean level density clears the bar
            double s = 0.0;
            for (u32 r = b0; r < b0 + 128; r++) s += (double)h[(size_t)k * m + order[r]];
            if (s / 128.0 < thr) break;
            G = b0 + 128;
        }
        if (G == 0) break;
        pl.G[k] = G;
        prev = G;
        L = k + 1;
    }
    if (L == 0) return SB_OK;
    pl.L = L;
    pl.ntiles = (mt->n + PL_TILE - 1) / PL_TILE;
    const u32 G1 = pl.G[0];
    std::vector<u32> hot(order.begin(), order.begin() + G1), hot_of(m, PL_NONE);
    for (u32 r = 0; r < G1; r++) hot_of[hot[r]] = r;
    SB_TRY(mt->hot_idx.alloc(G1));
    SB_TRY(mt->hot_of_gene.alloc(m));
    SB_CUDA(cudaMemcpyAsync(mt->hot_idx.p, hot.data(), G1 * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(mt->hot_of_gene.p, hot_of.data(), (size_t)m * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    for (u32 k = 0; k < L; k++) {
        const size_t words = std::max<size_t>(1, (size_t)pl.ntiles * (pl.G[k] / 32) * PL_TILE);
        SB_TRY(pl.bits[k].alloc(words));
        SB_CUDA(cudaMemsetAsync(pl.bits[k].p, 0, words * sizeof(u32), ctx->stream));
    }
    // ---- T-side units: (range of 1,024 ranks) x (up to three levels)
    std::vector<PlUnitT> ut;
    std::vector<double> cost;
    for (u32 g0 = 0; g0 < G1; g0 += PT_RANGE) {
        std::vector<u32> lv;
        for (u32 k = 0; k < L; k++)
            if (pl.G[k] > g0) lv.push_back(k);
        for (size_t i = 0; i < lv.size(); i += 3) {
            PlUnitT u;
            memset(&u, 0, sizeof(u));
            u.g0 = g0;
            double c = 0.0;
            for (size_t j = i; j < std::min(lv.size(), i + 3); j++) {
                const u32 genes = std::min(pl.G[lv[j]], g0 + PT_RANGE) - g0;  // multiple of 128
                u.lev[u.nlev] = lv[j];
                u.nkb[u.nlev] = genes / 32;
                u.nlev++;
                c += genes;
            }
            // the epilogue of a tile costs about as much as 100 ranks of MMA per level; with several levels it cannot overlap the
            // next tile's MMAs (one accumulator set)
            c += (u.nlev > 1 ? 250.0 : 100.0) * u.nlev;
            ut.push_back(u);
            cost.push_back(c);
        }
    }
    // work items: every unit's tiles in chunks of about equal cost, heaviest units first (the queue is drained in order by
    // persistent CTAs, so a long item never starts last); ~16 items per CTA keep the tail short
    {
        double total = 0.0;
        for (double c : cost) total += c * (double)pl.ntiles;
        const double target = std::max(1.0, total / ((double)ctx->sm_count * (double)std::max(1, ctx->plane_items_per_cta)));
        std::vector<u32> uo(ut.size());
        std::iota(uo.begin(), uo.end(), 0u);
        std::stable_sort(uo.begin(), uo.end(), [&](u32 x, u32 y) { return cost[x] > cost[y]; });
        std::vector<PlItem> items;
        for (u32 ui : uo) {
            const u64 per = std::max<u64>(1, (u64)(target / cost[ui] + 0.5));
            for (u64 t0 = 0; t0 < pl.ntiles; t0 += per) {
                PlItem it;
                it.unit = ui;
                it.t0 = (u32)t0;
                it.t1 = (u32)std::min<u64>(pl.ntiles, t0 + per);
                items.push_back(it);
            }
        }
        pl.n_units_t = (u32)ut.size();
        SB_TRY(pl.units_t.alloc(std::max<size_t>(1, ut.size()) * sizeof(PlUnitT)));
        if (!ut.empty()) SB_CUDA(cudaMemcpyAsync(pl.units_t.p, ut.data(), ut.size() * sizeof(PlUnitT), cudaMemcpyHostToDevice, ctx->stream));
        pl.n_items_t = (u32)items.size();
        pl.t_grid = (u32)std::min<size_t>((size_t)ctx->sm_count, std::max<size_t>(1, items.size()));
        SB_TRY(pl.items_t.alloc(std::max<size_t>(1, items.size()) * sizeof(PlItem)));
        if (!items.empty()) SB_CUDA(cudaMemcpyAsync(pl.items_t.p, items.data(), items.size() * sizeof(PlItem), cudaMemcpyHostToDevice, ctx->stream));
        SB_TRY(pl.counter.alloc(4));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));  // `items` is a host temporary
    }
    std::vector<u32> nc;
    u32 at = 0;
    // ---- N-side units: groups of 384 ranks; the active levels of a group are a prefix
    std::vector<PlUnitN> un;
    cost.clear();
    for (u32 g0 = 0; g0 < G1; g0 += PN_GROUP) {
        PlUnitN u;
        memset(&u, 0, sizeof(u));
        u.g0 = g0;
        double c = 0.0;
        for (u32 k = 0; k < L && pl.G[k] > g0; k++) {
            u.mt[k] = (std::min(pl.G[k], g0 + PN_GROUP) - g0) / 128;
            u.nlev = k + 1;
            c += u.mt[k] + 0.5;  // a stage costs its production (A words + the B copy) as well as its MMAs
        }
        un.push_back(u);
        cost.push_back(c);
    }
    {
        double total = 0.0;
        for (double c : cost) total += c * (double)pl.ntiles;
        const double target = std::max(1.0, total / ((double)ctx->sm_count * 10.0));
        std::vector<u32> uo(un.size());
        std::iota(uo.begin(), uo.end(), 0u);
        std::stable_sort(uo.begin(), uo.end(), [&](u32 x, u32 y) { return cost[x] > cost[y]; });
        std::vector<PlItem> items;
        for (u32 ui : uo) {
            // int32 accumulators: at most 2^24 cells per item (|digit| <= 128)
            const u64 per = std::min<u64>(std::max<u64>(1, (u64)(target / cost[ui] + 0.5)), (1u << 24) / PL_TILE);
            for (u64 t0 = 0; t0 < pl.ntiles; t0 += per) {
                PlItem it;
                it.unit = ui;
                it.t0 = (u32)t0;
                it.t1 = (u32)std::min<u64>(pl.ntiles, t0 + per);
                items.push_back(it);
            }
        }
        pl.n_items_n = (u32)items.size();
        pl.n_grid = (u32)std::min<size_t>((size_t)ctx->sm_count, std::max<size_t>(1, items.size()));
        SB_TRY(pl.items_n.alloc(std::max<size_t>(1, items.size()) * sizeof(PlItem)));
        if (!items.empty()) SB_CUDA(cudaMemcpyAsync(pl.items_n.p, items.data(), items.size() * sizeof(PlItem), cudaMemcpyHostToDevice, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));  // `items` is a host temporary
    }
    pl.n_units_n = (u32)un.size();
    SB_TRY(pl.units_n.alloc(std::max<size_t>(1, un.size()) * sizeof(PlUnitN)));
    SB_CUDA(cudaMemcpyAsync(pl.units_n.p, un.data(), un.size() * sizeof(PlUnitN), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));  // host temporaries
    pl.active = true;
    mt->gd = G1;
    if (TraceScope::on()) {
        fprintf(stderr, "[scanb200] planes: L=%u G =", L);
        for (u32 k = 0; k < L; k++) fprintf(stderr, " %u", pl.G[k]);
        fprintf(stderr, "  (T units %u / %u CTAs, N units %u / %u CTAs)\n", pl.n_units_t, pl.t_grid, pl.n_units_n, pl.n_grid);
    }
    return SB_OK;
}

// Splits the cell-major stream of a cell range into plane bits and the cold sparse entries (count pass when `out` is NULL,
// fill pass otherwise).  ptr is offset to the first cell of the range; cbase = its local cell index (a multiple of 128).
__global__ void k_split_planes(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, u64 cbase, const u32 *__restrict__ rank_of_gene,
                               PlDev pl, const u64 *__restrict__ new_ptr, u32 *__restrict__ counts, uint2 *__restrict__ out) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        const u64 s = ptr[c], e = ptr[c + 1];
        const u64 wpos = new_ptr ? new_ptr[c] : 0;
        const u64 cell = cbase + c, tile = cell / PL_TILE;
        const u32 cl = (u32)(cell % PL_TILE);
        u32 total = 0;
        for (u64 k0 = s; k0 < e; k0 += 32) {
            const u64 k = k0 + lane;
            const bool valid = k < e;
            const uint2 z = valid ? cm[k] : make_uint2(0, 0);
            const u32 r = valid ? rank_of_gene[z.x] : PL_NONE;
            const bool dense = valid && r != PL_NONE && z.y >= 1 && z.y <= pl.L && r < pl.G[z.y - 1];
            const bool cold = valid && !dense;
            if (out && dense) {
                const u32 lv = z.y - 1;
                atomicOr(pl.bits[lv] + ((tile * (pl.G[lv] / 32) + (r >> 5)) * PL_TILE + cl), 1u << (r & 31));
            }
            const unsigned mask = __ballot_sync(0xffffffffu, cold);
            if (out && cold) out[wpos + total + __popc(mask & ((1u << lane) - 1u))] = z;
            total += __popc(mask);
        }
        if (counts && lane == 0) counts[c] = total;
    }
}

int planes_split_launch(sb_mat *mt, u64 c0, u64 nc, const u64 *new_ptr, u32 *counts, uint2 *out) {
    sb_ctx *ctx = mt->ctx;
    if (nc == 0) return SB_OK;
    if (c0 % PL_TILE) return sb_fail(SB_ERR_UNSUPPORTED, "planes_split: range start %llu is not a multiple of 128", (unsigned long long)c0);
    u64 blocks = std::min<u64>((nc * 32 + 255) / 256, (u64)ctx->sm_count * 16);
    k_split_planes<<<(unsigned)std::max<u64>(1, blocks), 256, 0, ctx->stream>>>(mt->cm_ptr.p + c0, mt->cm.p, nc, c0, mt->hot_of_gene.p, make_pldev(mt),
                                                                                new_ptr, counts, out);
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

// ---------------------------------------------------------------- digit helpers
// Operand entries are split as they are: a finite entry of any magnitude is exact up to the 54-bit quantum of its column, and a NaN or
// +-inf makes the column's scale NaN, so that the plane part of that whole output column is NaN (include/scanb200.h, sb_nmat_dot).

// q (|q| <= 2^54) -> 7 balanced base-256 digits in [-128, 127]
__device__ __forceinline__ void digits7(long long q, signed char (&d)[PL_DIG]) {
#pragma unroll
    for (u32 s = 0; s < PL_DIG; s++) {
        const long long t = ((q + 128) & 255) - 128;
        d[s] = (signed char)t;
        q = (q - t) >> 8;
    }
}

// |v| as bits: non-negative doubles order like their bits, +inf above every finite value and NaN above +inf
__device__ __forceinline__ unsigned long long abs_bits(double v) { return (unsigned long long)__double_as_longlong(v) & 0x7FFFFFFFFFFFFFFFull; }

__device__ __forceinline__ void atomic_max_abs(unsigned long long *slot, double v) { atomicMax(slot, abs_bits(v)); }

// scale2[c] = 2^(e_c - PL_FIX) with |x| < 2^e_c for every entry of column c; ex[c] = PL_FIX - e_c.  e_c >= PL_FIX - 1074 keeps scale2 at
// least the smallest subnormal (a column below 2^-1020 is quantised to the spacing of doubles at zero).  A non-finite column maximum
// gives scale2 = NaN.
__global__ void k_pl_scales(const unsigned long long *__restrict__ colmax_bits, double *__restrict__ scale2, int *__restrict__ ex) {
    const u32 c = threadIdx.x;
    if (c >= PL_COLS) return;
    const double mx = __longlong_as_double((long long)colmax_bits[c]);
    if (!isfinite(mx)) {
        scale2[c] = __longlong_as_double(0x7FF8000000000000ll);
        ex[c] = 0;
        return;
    }
    int e = 0;
    if (mx > 0.0) frexp(mx, &e);
    e = max(e, PL_FIX - 1074);
    scale2[c] = ldexp(1.0, e - PL_FIX);
    ex[c] = PL_FIX - e;
}

// ---------------------------------------------------------------- T side: digit planes of Ys
__global__ void k_pl_colmax_t(const double *__restrict__ Y, u32 ldy, const u32 *__restrict__ hot_idx, const double *__restrict__ rs, u32 G1, u32 col0,
                              u32 wt, unsigned long long *__restrict__ colmax_bits) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G1 * PL_COLS) return;
    const u32 r = i / PL_COLS, c = i - r * PL_COLS;
    if (c >= wt) return;
    const u32 g = hot_idx[r];
    double v = Y[(size_t)g * ldy + col0 + c];
    if (rs) v *= rs[g];
    atomic_max_abs(&colmax_bits[c], v);
}

// Bd[range][k / 16][n / 8][n % 8][k % 16], k = rank % 1024, n = 7 c + s (digit s of column c); with `split` the second ten columns
// start at accumulator column 72 (a multiple of 8) so that each half of the epilogue warps reads its own aligned 72-column range
__global__ void k_pl_digits_t(const double *__restrict__ Y, u32 ldy, const u32 *__restrict__ hot_idx, const double *__restrict__ rs, u32 G1, u32 col0,
                              u32 wt, const int *__restrict__ ex, signed char *__restrict__ Bd, u32 split) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G1 * PL_COLS) return;
    const u32 r = i / PL_COLS, c = i - r * PL_COLS;
    const u32 g = hot_idx[r];
    double v = c < wt ? Y[(size_t)g * ldy + col0 + c] : 0.0;
    if (rs) v *= rs[g];
    const long long q = __double2ll_rn(ldexp(v, ex[c]));
    signed char d[PL_DIG];
    digits7(q, d);
    const u32 range = r / PT_RANGE, k = r - range * PT_RANGE;
    signed char *base = Bd + (size_t)range * PT_B_BYTES + (size_t)(k >> 4) * PT_KCHUNK_BYTES + (k & 15);
#pragma unroll
    for (u32 s = 0; s < PL_DIG; s++) {
        const u32 n = c * PL_DIG + s + ((split && c >= PL_COLS / 2) ? 2u : 0u);
        base[(size_t)(n >> 3) * 128 + (n & 7) * 16] = d[s];
    }
}

// ---------------------------------------------------------------- shared epilogue arithmetic
// acc[n], n = 7 c + s: digit s of column c.  value_c = sum_s acc_s 256^s.  Done on the FP64 pipe: int32 -> f64 by the
// exponent trick (one LOP3 + one DADD), digits 0..3 and 4..6 are summed exactly (both halves stay below 2^53 for
// |acc| <= 2^28), then hi * 2^32 + lo is the single rounding.
__device__ __forceinline__ double i32_to_f64(u32 r) {
    return __hiloint2double(0x43300000, (int)(r ^ 0x80000000u)) - 4503601774854144.0;  // 2^52 + 2^31
}

// reads the 144 accumulator columns of this thread's TMEM lane starting at `taddr` and returns the 20 recombined values
__device__ __forceinline__ void read_acc(u32 taddr, double (&val)[PL_COLS]) {
    double lo = 0.0, hi = 0.0;
#pragma unroll
    for (u32 cb = 0; cb < PL_NCOL; cb += 16) {
        u32 r[16];
        tmem_ld16(taddr + cb, r);
        tmem_ld_wait();
#pragma unroll
        for (u32 i = 0; i < 16; i++) {
            const u32 n = cb + i;  // compile-time after unrolling
            if (n < PL_COLS * PL_DIG) {
                const u32 c = n / PL_DIG, s = n - c * PL_DIG;
                const double d = i32_to_f64(r[i]);
                if (s == 0) lo = d;
                else if (s < 4) lo = fma(d, (double)(1u << (8 * s)), lo);
                else if (s == 4) hi = d;
                else hi = fma(d, (double)(1u << (8 * (s - 4))), hi);
                if (s == PL_DIG - 1) val[c] = fma(hi, 4294967296.0, lo);
            }
        }
    }
}

// res[c] += lk * value_c, straight from the accumulator (keeps the epilogue's register footprint small)
__device__ __forceinline__ void read_acc_fma(u32 taddr, double lk, double (&res)[PL_COLS]) {
    double lo = 0.0, hi = 0.0;
#pragma unroll
    for (u32 cb = 0; cb < PL_NCOL; cb += 16) {
        u32 r[16];
        tmem_ld16(taddr + cb, r);
        tmem_ld_wait();
#pragma unroll
        for (u32 i = 0; i < 16; i++) {
            const u32 n = cb + i;  // compile-time after unrolling
            if (n < PL_COLS * PL_DIG) {
                const u32 c = n / PL_DIG, s = n - c * PL_DIG;
                const double d = i32_to_f64(r[i]);
                if (s == 0) lo = d;
                else if (s < 4) lo = fma(d, (double)(1u << (8 * s)), lo);
                else if (s == 4) hi = d;
                else hi = fma(d, (double)(1u << (8 * (s - 4))), hi);
                if (s == PL_DIG - 1) res[c] = fma(lk, fma(hi, 4294967296.0, lo), res[c]);
            }
        }
    }
}

// Ten columns (70 digit columns, read as 4 x 16 + 8 accumulator columns from `taddr`): res[c] += lk * value_c.  The loads of the
// next chunk pair are in flight while the current pair is recombined (tcgen05.wait::ld waits for every outstanding load, so the
// chunks are issued two at a time).
__device__ __forceinline__ void read_acc_fma_half(u32 taddr, double lk, double (&res)[PL_COLS / 2]) {
    u32 ra[16], rb[16], rc[16], rd[16], re[8];
    double lo = 0.0, hi = 0.0;
    auto eat = [&](const u32 *r, u32 n0, u32 cnt) {
#pragma unroll
        for (u32 i = 0; i < cnt; i++) {
            const u32 n = n0 + i;  // compile-time after unrolling
            if (n < (PL_COLS / 2) * PL_DIG) {
                const u32 c = n / PL_DIG, sdig = n - c * PL_DIG;
                const double d = i32_to_f64(r[i]);
                if (sdig == 0) lo = d;
                else if (sdig < 4) lo = fma(d, (double)(1u << (8 * sdig)), lo);
                else if (sdig == 4) hi = d;
                else hi = fma(d, (double)(1u << (8 * (sdig - 4))), hi);
                if (sdig == PL_DIG - 1) res[c] = fma(lk, fma(hi, 4294967296.0, lo), res[c]);
            }
        }
    };
    tmem_ld16(taddr, ra);
    tmem_ld16(taddr + 16, rb);
    tmem_ld_wait();
    tmem_ld16(taddr + 32, rc);
    tmem_ld16(taddr + 48, rd);
    eat(ra, 0, 16);
    eat(rb, 16, 16);
    tmem_ld_wait();
    tmem_ld8(taddr + 64, re);
    eat(rc, 32, 16);
    eat(rd, 48, 16);
    tmem_ld_wait();
    eat(re, 64, 8);
}

// ---------------------------------------------------------------- k_planes_t
// Roles: warps 0-3 epilogue, warp 4 MMA issue, warps 5-20 producers, warp 21 scheduler.  The producers' refill latency
// (expand one sub-stage after its slot was freed) against the MMA work in flight in the ring decides the throughput: sixteen
// warps each own a 4 KB sub-slot (one MMA's A operand), four sub-slots make a stage.
// Two generations of the kernel (A/B through the option pl_variant bit 0; profiles/planes_r02_findings.md).
//   V = 0: warps 0-3 epilogue, 4 MMA issue, 5-12 producers, 13 item scheduler.
//   V = 1: what ncu showed of V = 0 at 400k cells -- (1) 17 % of all warp samples sit in the reload of the resident B block at a
//          unit change (a 21-iteration LDG -> STS loop per thread, one exposed L2 round trip each: ~16 us per change); (2) the four
//          epilogue warps are busy 70 % of the time: 3,600 cycles per (tile, level) job, a single warp per scheduler working
//          through nine dependent tcgen05.ld -> convert -> FMA chains, against 576-2,304 cycles of MMAs per job -- the epilogue,
//          not the tensor pipe (32 % busy), paces the kernel.  So: the B block arrives by bulk asynchronous copies (cp.async.bulk,
//          one thread, completion on an mbarrier); EIGHT epilogue warps, two per TMEM lane quarter (a warp may only touch lanes
//          32 (warp % 4) ..), each owning ten of the twenty columns, with the TMEM loads of the next chunk in flight while the
//          current one is recombined; descriptor low words carry the leading-byte-offset field so an MMA costs 7 issue slots
//          instead of 11.  Warps: 0-7 epilogue, 8 MMA, 9 item scheduler, 10-17 producers.
//          (Measured without effect and dropped: isolating the MMA warp on its scheduler, issuing two stages per election.)
template <int V> struct PtLayout;
template <> struct PtLayout<0> {
    static constexpr u32 WARPS = PL_EPI_WARPS + 1 + PT_PROD_WARPS + 1, EPI = PL_EPI_WARPS;
};
template <> struct PtLayout<1> {
    static constexpr u32 WARPS = 8 + 1 + 1 + PT_PROD_WARPS, EPI = 8;
};
struct PtShared {
    unsigned long long full[PT_NSTG], empty[PT_NSTG], tfull[3], tempty[3], item_full[2], item_empty[2], bload;
    u32 tmem;
    u32 item[2];  // work-item ring filled by the scheduler warp
    u32 pad;
    double scale2[PL_COLS];
};

// Persistent CTAs pull work items {unit, tile range} from a global queue (items are sized to ~equal cost and ordered by
// unit, so the resident B block is reloaded only when the unit changes).  The scheduler warp keeps a two-deep ring of item
// ids, so the roles run into the next item without draining the pipeline; only a change of unit (new B block) is a
// CTA-wide barrier.  Pipeline state carried across items: the sub-stage counter q (A ring) and the job counter j -- one
// job per (tile, level), accumulating into TMEM slot j % 3, so the epilogue of one level overlaps the MMAs of the next.
// Output: the CTA's 20 values per (unit, cell) go to part[unit][cell][20] with plain stores -- every (unit, tile) is
// produced exactly once -- and k_pl_reduce_t adds the units up (f64 reductions into T cost 1.3 cycles per lane on the
// LSU and were the bottleneck of the first version: 0.43 of 1.5 ms).
template <int V>
__global__ void __launch_bounds__(PtLayout<V>::WARPS * 32, 1)
k_planes_t(PlDev pl, const PlUnitT *__restrict__ units, const PlItem *__restrict__ items, u32 n_items, u32 *__restrict__ counter,
           const signed char *__restrict__ Bd, const double *__restrict__ scale2_g, const double *__restrict__ lk, u32 wt,
           double *__restrict__ part, u32 dbg) {
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char *sB = smem;
    unsigned char *sA = sB + PT_B_BYTES;
    PtShared *sh = reinterpret_cast<PtShared *>(sA + PT_NSTAGES * PT_STAGE_BYTES);
    using LY = PtLayout<V>;
    constexpr u32 PT_WARPS = LY::WARPS, PT_THREADS = LY::WARPS * 32, EPI = LY::EPI;  // roles: [0, EPI) epilogue, EPI MMA, EPI + 1 .. producers, last (V0) / EPI + 1 (V1) item scheduler
    constexpr u32 W_MMA = EPI, W_SCHED = V ? EPI + 1 : PT_WARPS - 1, W_PROD0 = V ? EPI + 2 : EPI + 1;
    const u32 tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const u32 full0 = smem_u32(sh->full), empty0 = smem_u32(sh->empty), tfull0 = smem_u32(sh->tfull), tempty0 = smem_u32(sh->tempty);
    const u32 ifull0 = smem_u32(sh->item_full), iempty0 = smem_u32(sh->item_empty), bload0 = smem_u32(&sh->bload);
    u32 breloads = 0;  // V1: bulk reloads of the B block so far (phase of `bload`)

    if (tid == 0) {
        for (u32 i = 0; i < PT_NSTG; i++) {
            mbar_init(full0 + 8 * i, PT_SUB);  // one arrival per producer warp of the stage
            mbar_init(empty0 + 8 * i, 1);
        }
        for (u32 i = 0; i < 3; i++) {
            mbar_init(tfull0 + 8 * i, 1);
            mbar_init(tempty0 + 8 * i, EPI);
        }
        mbar_init(bload0, 1);
        for (u32 i = 0; i < 2; i++) {
            mbar_init(ifull0 + 8 * i, 1);
            mbar_init(iempty0 + 8 * i, PT_WARPS - 1);  // every consumer warp
        }
        mbar_init_fence();
    }
    if (warp == 0) tmem_alloc_512(smem_u32(&sh->tmem));
    if (tid < PL_COLS) sh->scale2[tid] = scale2_g[tid];
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const u32 tmem = sh->tmem;
    const u32 sA_addr = smem_u32(sA), sB_addr = smem_u32(sB);
    const u32 idesc = instr_desc_i8(PL_TILE, PL_NCOL, false, false);
    const uint64_t da_hi = smem_desc(0, PL_TILE * 16, 128), db_hi = smem_desc(0, PT_KCHUNK_BYTES, 128);
    const u64 n_pad = pl.ntiles * PL_TILE;
    const bool scheduler = warp == W_SCHED;

    u32 q = 0;      // 64-gene sub-stages before this item (producers) / issued so far (MMA)
    u32 job = 0;    // (tile, level) accumulation jobs so far
    u32 fills = 0;  // producer: fills of my sub-slot
    u32 cur_unit = 0xFFFFFFFFu;
    u32 g0 = 0, nlev = 0, nkb0 = 0, nkb1 = 0, nkb2 = 0, lev0 = 0, lev1 = 0, lev2 = 0, S = 2;

    for (u32 round = 0;; round++) {
        const u32 rs = round & 1u;
        u32 it;
        if (scheduler) {
            if (round >= 2) mbar_wait(iempty0 + 8 * rs, ((round >> 1) - 1) & 1u);
            it = 0;
            if (lane == 0) {
                it = atomicAdd(counter, 1u);
                sh->item[rs] = it;
            }
            it = __shfl_sync(0xffffffffu, it, 0);
            __syncwarp();
            if (lane == 0) mbar_arrive(ifull0 + 8 * rs);
        } else {
            mbar_wait(ifull0 + 8 * rs, (round >> 1) & 1u);
            it = sh->item[rs];
            __syncwarp();
            if (lane == 0) mbar_arrive(iempty0 + 8 * rs);
        }
        if (it >= n_items) break;
        const PlItem item = items[it];
        if (item.unit != cur_unit) {
            // new B block: drain (all MMAs that read the old block have completed once every role is here), reload, go on
            fence_before_sync();
            __syncthreads();
            fence_after_sync();
            const PlUnitT un = units[item.unit];
            cur_unit = item.unit;
            g0 = un.g0;
            nlev = un.nlev;
            nkb0 = un.nkb[0];
            nkb1 = nlev > 1 ? un.nkb[1] : 0;
            nkb2 = nlev > 2 ? un.nkb[2] : 0;
            lev0 = un.lev[0];
            lev1 = nlev > 1 ? un.lev[1] : 0;
            lev2 = nlev > 2 ? un.lev[2] : 0;
            S = (nkb0 + nkb1 + nkb2) / PT_WORDS;  // sub-stages per tile, level-major: [level 0 | level 1 | level 2]
            if (V == 1) {
                // one thread starts nine 16 KB bulk copies (the TMA engine's 1-D form); everybody waits on their byte count
                if (tid == 0) {
                    mbar_expect_tx(bload0, PT_B_BYTES);
                    const signed char *src = Bd + (size_t)(g0 / PT_RANGE) * PT_B_BYTES;
#pragma unroll 1
                    for (u32 o = 0; o < PT_B_BYTES; o += 16384u) bulk_g2s(sB_addr + o, src + o, 16384u, bload0);
                    mbar_arrive(bload0);
                }
                mbar_wait(bload0, breloads & 1u);
                breloads++;
            } else {
                const uint4 *src = reinterpret_cast<const uint4 *>(Bd + (size_t)(g0 / PT_RANGE) * PT_B_BYTES);
                uint4 *dst = reinterpret_cast<uint4 *>(sB);
                for (u32 i = tid; i < PT_B_BYTES / 16; i += PT_THREADS) dst[i] = src[i];
                fence_async_smem();
                __syncthreads();
            }
        }
        const u64 t0 = item.t0, t1 = item.t1;

        if (V == 1 && warp < EPI) {
            // ===== epilogue, V1: warp w reads TMEM lanes 32 (w % 4) .. of columns [72 (w / 4), 72 (w / 4) + 72): ten columns of 32 cells
            const u32 quarter = warp & 3u, half = warp >> 2;
            const u32 row = quarter * 32 + lane;
            double *pu = part + (size_t)item.unit * n_pad * PL_COLS + half * (PL_COLS / 2);
            for (u64 tile = t0; tile < t1; tile++) {
                const u64 cell = tile * PL_TILE + row;
                double res[PL_COLS / 2];
#pragma unroll
                for (u32 j = 0; j < PL_COLS / 2; j++) res[j] = 0.0;
                double L0 = 0.0, L1 = 0.0, L2 = 0.0;
                if (cell < pl.n) {  // L_c(level) from the per-cell table written by sb_normalize
                    const double *lc = lk + cell * PL_MAX_LEVELS;
                    L0 = lc[lev0];
                    if (nlev > 1) L1 = lc[lev1];
                    if (nlev > 2) L2 = lc[lev2];
                }
                for (u32 a = 0; a < nlev; a++, job++) {
                    const u32 slot = job % 3u;
                    mbar_wait(tfull0 + 8 * slot, (job / 3u) & 1u);
                    fence_after_sync();
                    if (!(dbg & 2u)) read_acc_fma_half(tmem + ((quarter * 32u) << 16) + slot * PL_NCOL + half * 72u, a == 0 ? L0 : (a == 1 ? L1 : L2), res);
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tempty0 + 8 * slot);
                }
                if (!(dbg & 1u)) {
                    double2 *o = reinterpret_cast<double2 *>(pu + cell * PL_COLS);
#pragma unroll
                    for (u32 j = 0; j < PL_COLS / 2; j += 2)
                        o[j >> 1] = make_double2(res[j] * sh->scale2[half * (PL_COLS / 2) + j], res[j + 1] * sh->scale2[half * (PL_COLS / 2) + j + 1]);
                }
            }
        } else if (warp < EPI) {
            // ===== epilogue: TMEM -> registers -> f64 -> partial output (one thread per cell row)
            const u32 row = warp * 32 + lane;
            double *pu = part + (size_t)item.unit * n_pad * PL_COLS;
            for (u64 tile = t0; tile < t1; tile++) {
                const u64 cell = tile * PL_TILE + row;
                double res[PL_COLS];
#pragma unroll
                for (u32 j = 0; j < PL_COLS; j++) res[j] = 0.0;
                double L0 = 0.0, L1 = 0.0, L2 = 0.0;
                if (cell < pl.n) {  // L_c(level) from the per-cell table written by sb_normalize
                    const double *lc = lk + cell * PL_MAX_LEVELS;
                    L0 = lc[lev0];
                    if (nlev > 1) L1 = lc[lev1];
                    if (nlev > 2) L2 = lc[lev2];
                }
                for (u32 a = 0; a < nlev; a++, job++) {
                    const u32 slot = job % 3u;
                    mbar_wait(tfull0 + 8 * slot, (job / 3u) & 1u);
                    fence_after_sync();
                    if (!(dbg & 2u)) read_acc_fma(tmem + ((warp * 32u) << 16) + slot * PL_NCOL, a == 0 ? L0 : (a == 1 ? L1 : L2), res);
                    fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(tempty0 + 8 * slot);  // this warp's quarter of the accumulator is free
                }
                if (!(dbg & 1u)) {  // rows of a tile are adjacent: a warp writes 32 x 160 contiguous bytes
                    double2 *o = reinterpret_cast<double2 *>(pu + cell * PL_COLS);
#pragma unroll
                    for (u32 j = 0; j < PL_COLS; j += 2) o[j >> 1] = make_double2(res[j] * sh->scale2[j], res[j + 1] * sh->scale2[j + 1]);
                }
            }
        } else if (warp == W_MMA) {
            // ===== MMA issue.  The warp runs the loops converged, every value warp-uniform, and only the tensor-core instructions
            // are predicated on an elected lane: that keeps descriptors and addresses in uniform registers (UIADD3 / ULOP3 +
            // UTCIMMA).  Electing a lane around the whole loop instead makes the compiler wrap each UTCIMMA in an ELECT /
            // 5 x R2UR.BROADCAST / branch loop -- ~90 instructions per 4-MMA stage, more than the 288 cycles the MMAs take.
            {
                const u32 a16 = sA_addr >> 4, b16 = sB_addr >> 4;
                // V = 1: the low descriptor words carry the leading-byte-offset field (bits 16-29; the 14-bit address field below
                // it never carries into it), so a descriptor is one add away from the previous one and the high word is an immediate
                const u32 a16x = a16 + ((PL_TILE * 16u >> 4) << 16), b16x = b16 + ((PT_KCHUNK_BYTES >> 4) << 16);
                auto level = [&](u32 nkb) {
                    const u32 slot = job % 3u;
                    if (job >= 3u) {
                        mbar_spin(tempty0 + 8 * slot, (job / 3u - 1u) & 1u);
                        fence_after_sync();
                    }
                    const u32 acc = tmem + slot * PL_NCOL;
                    u32 kb = 0;
                    if (V == 1) {
                        for (; kb < nkb; kb += PT_SUB * PT_WORDS) {
                            const u32 sg = q / PT_SUB, ss = sg & (PT_NSTG - 1);
                            mbar_spin(full0 + 8 * ss, (sg / PT_NSTG) & 1u);
                            fence_after_sync();
                            const u32 alo = a16x + ss * (PT_SUB * PT_STAGE_BYTES >> 4), blo = b16x + kb * (2 * PT_KCHUNK_BYTES >> 4);
                            if (elect_one()) {
#pragma unroll
                                for (u32 t = 0; t < PT_SUB * PT_WORDS; t++)
                                    mma_i8_lo<0x4008u, 0x4008u>(acc, alo + t * (PL_TILE * 32 >> 4), blo + t * (2 * PT_KCHUNK_BYTES >> 4), idesc, kb | t);
                                commit(empty0 + 8 * ss);
                            }
                            __syncwarp();
                            q += PT_SUB;
                        }
                    }
                    for (; kb < nkb; kb += PT_SUB * PT_WORDS) {  // kb counts 32-gene blocks (one MMA each)
                        const u32 sg = q / PT_SUB, ss = sg & (PT_NSTG - 1);
                        mbar_spin(full0 + 8 * ss, (sg / PT_NSTG) & 1u);
                        fence_after_sync();
                        const u32 alo = a16 + ss * (PT_SUB * PT_STAGE_BYTES >> 4), blo = b16 + kb * (2 * PT_KCHUNK_BYTES >> 4);
                        if (elect_one()) {
#pragma unroll
                            for (u32 t = 0; t < PT_SUB * PT_WORDS; t++)  // K = 32 per MMA = two 16-gene core-matrix columns (4 KB of A)
                                mma_i8(acc, da_hi | (alo + t * (PL_TILE * 32 >> 4)), db_hi | (blo + t * (2 * PT_KCHUNK_BYTES >> 4)), idesc, kb | t);
                            commit(empty0 + 8 * ss);  // the stage is reusable once these MMAs have read it
                        }
                        __syncwarp();
                        q += PT_SUB;
                    }
                    if (elect_one()) commit(tfull0 + 8 * slot);  // this level's accumulator is complete
                    __syncwarp();
                    job++;
                };
                for (u64 tile = t0; tile < t1; tile++) {
                    level(nkb0);
                    if (nlev > 1) level(nkb1);
                    if (nlev > 2) level(nkb2);
                }
            }
        } else if (!scheduler) {
            // ===== producers: plane words -> 0/1 int8 A tiles (K-major core matrices: [16-gene chunk][cell / 8][cell % 8][16 B])
            // warp p fills sub-slot p: the sub-stages (PT_WORDS x 32 genes of one level) with global index = p (mod PT_NSTAGES)
            const u32 p = warp - W_PROD0;
            const u32 G0 = pl.G[lev0] >> 5, G1w = pl.G[lev1] >> 5, G2w = pl.G[lev2] >> 5;
            const u32 *bits0 = pl.bits[lev0], *bits1 = pl.bits[lev1], *bits2 = pl.bits[lev2];
            const u32 s0 = nkb0 / PT_WORDS, s1 = nkb1 / PT_WORDS;  // sub-stages of levels 0, 1 per tile
            u64 tile = t0;
            u32 i = (p + PT_NSTAGES - (q & (PT_NSTAGES - 1))) & (PT_NSTAGES - 1);  // my first sub-stage inside this item
            while (i >= S && tile < t1) {
                i -= S;
                tile++;
            }
            auto load_words = [&](u64 tl, u32 ii, u32 (&w)[4 * PT_WORDS]) {  // ii: sub-stage inside the tile, level-major
                const bool in1 = ii >= s0, in2 = ii >= s0 + s1;
                const u32 sb = ii - (in2 ? s0 + s1 : (in1 ? s0 : 0u));
                const u32 Gw = in2 ? G2w : (in1 ? G1w : G0);
                const u32 *bp = in2 ? bits2 : (in1 ? bits1 : bits0);
                const u32 *base = bp + ((size_t)tl * Gw + (g0 >> 5) + sb * PT_WORDS) * PL_TILE + lane;
#pragma unroll
                for (u32 j = 0; j < PT_WORDS; j++)
#pragma unroll
                    for (u32 c4 = 0; c4 < 4; c4++) w[j * 4 + c4] = __ldg(base + (size_t)j * PL_TILE + c4 * 32);
            };
            // L2 prefetch: the plane words of a (tile, level) for this range are contiguous (nkb KB); when this warp first touches
            // a tile it pulls its eighth of the tile two ahead towards L2
            auto prefetch_tile = [&](u64 tl) {
                if (tl >= t1) return;
                const u32 line = p * (128 / PT_NSTAGES) + lane;  // 128-byte lines; a full range has 128 per level (4 per 32-gene block)
                if (lane < 128 / PT_NSTAGES) {
                    if (line < nkb0 * 4) prefetch_l2(bits0 + ((size_t)tl * G0 + (g0 >> 5)) * PL_TILE + line * 32);
                    if (line < nkb1 * 4) prefetch_l2(bits1 + ((size_t)tl * G1w + (g0 >> 5)) * PL_TILE + line * 32);
                    if (line < nkb2 * 4) prefetch_l2(bits2 + ((size_t)tl * G2w + (g0 >> 5)) * PL_TILE + line * 32);
                }
            };
            u32 cur[4 * PT_WORDS], nxt[4 * PT_WORDS];
            bool live = tile < t1;
            if (live) {
                prefetch_tile(tile + 1);
                prefetch_tile(tile + 2);
                load_words(tile, i, cur);
            }
            const u32 st = sA_addr + p * PT_STAGE_BYTES + lane * 16;
            while (live) {
                // my next sub-stage: prefetch its words before expanding the current ones
                u64 ntile = tile;
                u32 ni = i + PT_NSTAGES;
                while (ni >= S && ntile < t1) {
                    ni -= S;
                    ntile++;
                }
                const bool more = ntile < t1;
                if (more) load_words(ntile, ni, nxt);
                if (ntile != tile) prefetch_tile(ntile + 2);
                if (V == 1) {
                    // the refill of a freed slot is on the critical path of the ring (microbenchmarks: 190 cycles from the last MMA to
                    // the `empty` phase, 125-215 per barrier hop, against 1,152 cycles of MMAs in the whole ring): the expansion
                    // arithmetic happens BEFORE the wait, into registers, and only the sixteen stores follow it
                    // (the first 32-gene word group only: all sixteen vectors would need 64 registers and spill under the 96 this CTA
                    // size allows; the second group is expanded after the wait, while the first group's stores drain)
                    uint4 ex[8];
#pragma unroll
                    for (u32 c4 = 0; c4 < 4; c4++) expand_bits32(cur[c4], ex[2 * c4], ex[2 * c4 + 1]);
                    if (fills > 0) mbar_wait(empty0 + 8 * (p / PT_SUB), (fills - 1) & 1u);
                    if (!(dbg & 4u)) {
#pragma unroll
                        for (u32 c4 = 0; c4 < 4; c4++) {
                            st_shared_v4(st + c4 * 512, ex[2 * c4]);
                            st_shared_v4(st + (PL_TILE * 16) + c4 * 512, ex[2 * c4 + 1]);
                        }
#pragma unroll
                        for (u32 j = 1; j < PT_WORDS; j++)
#pragma unroll
                            for (u32 c4 = 0; c4 < 4; c4++) {
                                uint4 lo, hi;
                                expand_bits32(cur[j * 4 + c4], lo, hi);
                                st_shared_v4(st + (2 * j) * (PL_TILE * 16) + c4 * 512, lo);
                                st_shared_v4(st + (2 * j + 1) * (PL_TILE * 16) + c4 * 512, hi);
                            }
                    }
                } else {
                if (fills > 0) mbar_wait(empty0 + 8 * (p / PT_SUB), (fills - 1) & 1u);
                if (!(dbg & 4u))
#pragma unroll
                    for (u32 j = 0; j < PT_WORDS; j++)
#pragma unroll
                        for (u32 c4 = 0; c4 < 4; c4++) {
                            uint4 lo, hi;
                            expand_bits32(cur[j * 4 + c4], lo, hi);
                            st_shared_v4(st + (2 * j) * (PL_TILE * 16) + c4 * 512, lo);
                            st_shared_v4(st + (2 * j + 1) * (PL_TILE * 16) + c4 * 512, hi);
                        }
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(full0 + 8 * (p / PT_SUB));
                fills++;
                tile = ntile;
                i = ni;
                live = more;
                if (more) {
#pragma unroll
                    for (u32 c = 0; c < 4 * PT_WORDS; c++) cur[c] = nxt[c];
                }
            }
            q += (u32)(t1 - t0) * S;
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc_512(tmem);
}

// T[c, col0 + j] += sum over units of part[u][c][j]  (+ l1[c] * t1[c][j]: the sparse gather's run sums in units of L_c(1), when deferred)
__global__ void k_pl_reduce_t(const double *__restrict__ part, u32 n_units, u64 n, u64 n_pad, u32 col0, u32 wt, double *__restrict__ out, u32 ldo,
                              const double *__restrict__ t1, const double *__restrict__ l1) {
    const u64 total = n * (PL_COLS / 2);
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (u64)gridDim.x * blockDim.x) {
        const u64 c = i / (PL_COLS / 2);
        const u32 j = (u32)(i - c * (PL_COLS / 2)) * 2;
        if (j >= wt) continue;
        double2 s = make_double2(0.0, 0.0);
        for (u32 u = 0; u < n_units; u++) {
            const double2 v = *reinterpret_cast<const double2 *>(part + ((size_t)u * n_pad + c) * PL_COLS + j);
            s.x += v.x;
            s.y += v.y;
        }
        if (t1) {  // a cell without sparse entries adds nothing: a zero-total cell has L_c(1) = inf, and inf * 0 would be NaN
            const double2 v = *reinterpret_cast<const double2 *>(t1 + c * PL_COLS + j);
            const double f = l1[c];
            if (v.x != 0.0) s.x = fma(f, v.x, s.x);
            if (v.y != 0.0) s.y = fma(f, v.y, s.y);
        }
        double *o = out + c * (size_t)ldo + col0 + j;
        o[0] += s.x;
        if (j + 1 < wt) o[1] += s.y;
    }
}

// ---------------------------------------------------------------- N side: digit rows of L_c(k) . X[c,:]
// mode 0: value_j = L_c(k) * X[c, col0 + j]; mode 1 (moments): value_0 = L_c(k), value_1 = L_c(k)^2
__global__ void k_pl_colmax_n(const double *__restrict__ X, u32 ldx, u64 n, const double *__restrict__ lk, u32 Ltop, u32 col0, u32 wt,
                              int mode, unsigned long long *__restrict__ colmax_bits) {
    unsigned long long mx[PL_COLS];  // abs_bits: the maximum keeps a NaN (fmax would drop it)
#pragma unroll
    for (u32 j = 0; j < PL_COLS; j++) mx[j] = 0ull;
    for (u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (u64)gridDim.x * blockDim.x) {
        const double l = lk[c * PL_MAX_LEVELS + Ltop - 1];  // L_c(k) grows with k: the top level bounds all
        if (mode == 1) {
            mx[0] = max(mx[0], abs_bits(l));
            mx[1] = max(mx[1], abs_bits(l * l));
        } else {
#pragma unroll
            for (u32 j = 0; j < PL_COLS; j++)
                if (j < wt) mx[j] = max(mx[j], abs_bits(l * X[c * (size_t)ldx + col0 + j]));
        }
    }
#pragma unroll
    for (u32 j = 0; j < PL_COLS; j++) {
        unsigned long long v = mx[j];
        for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
        if ((threadIdx.x & 31) == 0 && v != 0ull) atomicMax(&colmax_bits[j], v);
    }
}

// Bn[level][cell / 8][n / 16][cell % 8][n % 16] over the padded cells (zero rows beyond n): one thread per (cell, level)
__global__ void k_pl_digits_n(const double *__restrict__ X, u32 ldx, u64 n, u64 n_pad, const double *__restrict__ lk, u32 L, u32 col0,
                              u32 wt, int mode, const int *__restrict__ ex, signed char *__restrict__ Bn) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad * L) return;
    const u32 lv = (u32)(i / n_pad);
    const u64 c = i - (u64)lv * n_pad;
    u32 pk[PL_NCOL / 4];
#pragma unroll
    for (u32 t = 0; t < PL_NCOL / 4; t++) pk[t] = 0u;
    if (c < n) {
        const double l = lk[c * PL_MAX_LEVELS + lv];
#pragma unroll
        for (u32 j = 0; j < PL_COLS; j++) {
            double v = 0.0;
            if (mode == 1) v = j == 0 ? l : (j == 1 ? l * l : 0.0);
            else if (j < wt) v = l * X[c * (size_t)ldx + col0 + j];
            const long long q = __double2ll_rn(ldexp(v, ex[j]));
            signed char d[PL_DIG];
            digits7(q, d);
#pragma unroll
            for (u32 s = 0; s < PL_DIG; s++) {
                const u32 nn = j * PL_DIG + s;  // compile-time
                pk[nn >> 2] |= (u32)(unsigned char)d[s] << (8 * (nn & 3));
            }
        }
    }
    uint4 *dst = reinterpret_cast<uint4 *>(Bn + ((size_t)lv * (n_pad / 8) + (c >> 3)) * PN_CELLGRP_BYTES + (c & 7) * 16);
#pragma unroll
    for (u32 t = 0; t < PL_NCOL / 16; t++) dst[t * 8] = make_uint4(pk[4 * t], pk[4 * t + 1], pk[4 * t + 2], pk[4 * t + 3]);  // chunks are 128 B apart
}

// ---------------------------------------------------------------- k_planes_n
struct PnShared {
    unsigned long long full[PN_NSTG], empty[PN_NSTG], tfull;
    u32 tmem;
    u32 item[2];
    u32 pad;
    double scale2[PL_COLS];
};

// out[gene * row_stride + (col0 + j) * col_stride] += value
// Persistent CTAs pull work items {group of 384 ranks, range of cell tiles} from a global queue (about equal cost each); an item
// ends with its epilogue (the accumulators are reused by the next item), so the CTA-wide barrier between items costs nothing extra.
// V = 1: twelve producer warps (ncu: the N side waits on its producers -- 114 polls of the `full` barrier per stage by the MMA
// warp, producers busy 80 % of the time) and the digit rows of a sub-stage (4,608 contiguous bytes) arrive by one bulk
// asynchronous copy (cp.async.bulk, completion counted on the stage's `full` barrier) instead of 9 LDG.128 + 9 STS.128 per lane.
template <int V>
__global__ void __launch_bounds__((PL_EPI_WARPS + 1 + (V ? 12 : 8)) * 32, 1)
k_planes_n(PlDev pl, const PlUnitN *__restrict__ units, const PlItem *__restrict__ items, u32 n_items, u32 *__restrict__ counter,
           const signed char *__restrict__ Bn, u64 n_pad, const double *__restrict__ scale2_g, const u32 *__restrict__ hot_idx, u32 col0, u32 wt,
           double *__restrict__ out, u64 row_stride, u64 col_stride) {
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char *sS = smem;  // PN_NSTAGES sub-slots: [A: 3 M tiles x 4,096 | B: 4,608]
    PnShared *sh = reinterpret_cast<PnShared *>(sS + PN_NSTAGES * PN_STAGE_BYTES);
    const u32 tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const u32 full0 = smem_u32(sh->full), empty0 = smem_u32(sh->empty), tfull0 = smem_u32(&sh->tfull);
    constexpr u32 PW = V ? 12u : 8u;  // producer warps
    if (tid == 0) {
        for (u32 i = 0; i < PN_NSTG; i++) {
            mbar_init(full0 + 8 * i, PN_SUB);  // one arrival per producer warp of the stage
            mbar_init(empty0 + 8 * i, 1);
        }
        mbar_init(tfull0, 1);
        mbar_init_fence();
        sh->item[0] = atomicAdd(counter, 1u);
    }
    if (warp == 0) tmem_alloc_512(smem_u32(&sh->tmem));
    if (tid < PL_COLS) sh->scale2[tid] = scale2_g[tid];
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const u32 tmem = sh->tmem;
    const u32 sS_addr = smem_u32(sS);
    const u32 idesc = instr_desc_i8(128, PL_NCOL, true, true);
    const uint64_t da_hi = smem_desc(0, 128, 512);               // MN-major A: lbo = next 8 cells, sbo = next 16 genes
    const uint64_t db_hi = smem_desc(0, PN_CELLGRP_BYTES, 128);  // MN-major B: lbo = next 8 cells, sbo = next 16 digit columns

    u32 sg = 0;  // stages issued (MMA) / sub-stages before this item (producers: Q0)
    u32 Q0 = 0;
    for (u32 round = 0;; round++) {
        const u32 it = sh->item[round & 1];
        if (it >= n_items) break;
        if (tid == 0) sh->item[(round + 1) & 1] = atomicAdd(counter, 1u);  // visible after the barrier that ends this round
        const PlItem item = items[it];
        const PlUnitN un = units[item.unit];
        const u32 nlev = un.nlev, g0w = un.g0 >> 5;
        u32 mt_pack = 0;  // four bits per level: M tiles of the level inside this group
        for (u32 k = 0; k < nlev; k++) mt_pack |= un.mt[k] << (4 * k);
        const u64 t_begin = item.t0, t_end = item.t1;

        if (warp < PL_EPI_WARPS) {
            // ===== epilogue (once per item): TMEM lanes = gene rows of an M tile
            mbar_wait_sleep(tfull0, round & 1u);
            fence_after_sync();
            const u32 row = warp * 32 + lane;
            for (u32 mtile = 0; mtile < (mt_pack & 15u); mtile++) {
                double val[PL_COLS];
                read_acc(tmem + ((warp * 32u) << 16) + mtile * PL_NCOL, val);
                const u32 g = hot_idx[un.g0 + mtile * 128 + row];
                double *o = out + (size_t)g * row_stride;
#pragma unroll
                for (u32 j = 0; j < PL_COLS; j++) {
                    const double r = val[j] * sh->scale2[j];  // NaN in every row of a column whose scale is NaN, zero or not
                    if (j < wt && r != 0.0) atomicAdd(o + (size_t)(col0 + j) * col_stride, r);
                }
            }
        } else if (warp == PL_EPI_WARPS) {
            // ===== MMA issue: converged warp, uniform values, an elected lane only around the tensor-core instructions (see k_planes_t);
            // a stage = a whole 128-cell tile of one level = four K steps x up to three M tiles
            const u32 s16 = sS_addr >> 4;
            u32 started = 0;  // bit mtile: the accumulator has been written
            for (u64 tile = t_begin; tile < t_end; tile++) {
                u32 mtp = mt_pack;
                for (u32 k = 0; k < nlev; k++, mtp >>= 4, sg++) {
                    const u32 slot = sg % PN_NSTG;
                    mbar_spin(full0 + 8 * slot, (sg / PN_NSTG) & 1u);
                    fence_after_sync();
                    const u32 nmt = mtp & 15u;
                    if (V == 1) {
                        if (elect_one()) {
#pragma unroll
                            for (u32 ks = 0; ks < PN_SUB; ks++) {
                                const u32 alo = s16 + (slot * PN_SUB + ks) * (PN_STAGE_BYTES >> 4) + ((128u >> 4) << 16);
                                const u32 blo = s16 + (slot * PN_SUB + ks) * (PN_STAGE_BYTES >> 4) + (PN_A_BYTES >> 4) + ((PN_CELLGRP_BYTES >> 4) << 16);
                                mma_i8_lo<0x4020u, 0x4008u>(tmem, alo, blo, idesc, (started & 1u) | ks);
                                if (nmt > 1) mma_i8_lo<0x4020u, 0x4008u>(tmem + PL_NCOL, alo + 256, blo, idesc, ((started >> 1) & 1u) | ks);
                                if (nmt > 2) mma_i8_lo<0x4020u, 0x4008u>(tmem + 2 * PL_NCOL, alo + 512, blo, idesc, ((started >> 2) & 1u) | ks);
                            }
                            commit(empty0 + 8 * slot);
                        }
                    } else if (elect_one()) {
#pragma unroll
                        for (u32 ks = 0; ks < PN_SUB; ks++) {
                            const u32 alo = s16 + (slot * PN_SUB + ks) * (PN_STAGE_BYTES >> 4);
                            const uint64_t db = db_hi | (alo + (PN_A_BYTES >> 4));
                            mma_i8(tmem, da_hi | alo, db, idesc, (started & 1u) | ks);
                            if (nmt > 1) mma_i8(tmem + PL_NCOL, da_hi | (alo + 256), db, idesc, ((started >> 1) & 1u) | ks);
                            if (nmt > 2) mma_i8(tmem + 2 * PL_NCOL, da_hi | (alo + 512), db, idesc, ((started >> 2) & 1u) | ks);
                        }
                        commit(empty0 + 8 * slot);
                    }
                    __syncwarp();
                    started |= (1u << nmt) - 1u;
                }
            }
            if (elect_one()) commit(tfull0);
            __syncwarp();
        } else {
            // ===== producers: sub-stage = (32-cell K step, level): A tiles [M tile][16-gene chunk (8)][cell / 8 (4)][cell % 8][16 B] + B
            // digit rows.  Sub-stage Q of the CTA (tile-major, then level, then K step) goes to ring slot Q % 12, filled by warp Q % 8.
            const u32 p = warp - (PL_EPI_WARPS + 1);
            const u32 per_tile = PN_SUB * nlev;
            u32 cur[12], nxt[12];
            u64 tile = t_begin;
            u32 r = (p + PW - (Q0 % PW)) % PW;  // my first sub-stage inside this item: r = k * 4 + ks
            u32 Q = Q0 + r;                                                         // its global index
            while (r >= per_tile && tile < t_end) {
                r -= per_tile;
                tile++;
            }
            auto load_words = [&](u64 tl, u32 ks, u32 k, u32 (&w)[12]) {
                const u32 nw = ((mt_pack >> (4 * k)) & 15u) * 4;
                const u32 *base = pl.bits[k] + ((size_t)tl * (pl.G[k] >> 5) + g0w) * PL_TILE + ks * 32 + lane;
#pragma unroll
                for (u32 j = 0; j < 12; j++) w[j] = (j < nw) ? __ldg(base + (size_t)j * PL_TILE) : 0u;
            };
            // L2 prefetch two tiles ahead: per level the group's plane words (mt x 2 KB) and the digit rows of the tile's 128
            // cells (18 KB) are contiguous; each producer warp pulls its share when it first touches a tile
            auto prefetch_tile = [&](u64 tl) {
                if (tl >= t_end) return;
                for (u32 kk = 0; kk < nlev; kk++) {
                    const u32 alines = ((mt_pack >> (4 * kk)) & 15u) * 16;  // 128-byte lines of A words
                    const u32 line = p * 32 + lane;                          // 0..255: A lines first, then the 144 B lines
                    if (line < alines) prefetch_l2(pl.bits[kk] + ((size_t)tl * (pl.G[kk] >> 5) + g0w) * PL_TILE + line * 32);
                    else if (line - alines < 144) prefetch_l2(Bn + ((size_t)kk * (n_pad / 8) + tl * (PL_TILE / 8)) * PN_CELLGRP_BYTES + (size_t)(line - alines) * 128);
                }
            };
            bool live = tile < t_end;
            u32 ks = r & 3u, k = r >> 2;
            if (live) {
                prefetch_tile(tile + 1);
                prefetch_tile(tile + 2);
                load_words(tile, ks, k, cur);
            }
            while (live) {
                u64 ntile = tile;
                u32 nr = r + PW;
                while (nr >= per_tile) {
                    nr -= per_tile;
                    ntile++;
                }
                const bool more = ntile < t_end;
                const u32 nks = nr & 3u, nk = nr >> 2;
                if (more) load_words(ntile, nks, nk, nxt);
                if (ntile != tile) prefetch_tile(ntile + 2);
                // B rows of these 32 cells at level k (contiguous 4,608 bytes in Bn)
                const uint4 *bsrc = reinterpret_cast<const uint4 *>(Bn + ((size_t)k * (n_pad / 8) + (tile * PL_TILE + ks * 32) / 8) * PN_CELLGRP_BYTES);
                uint4 bv[V ? 1 : PN_B_BYTES / 16 / 32];
                if (V == 0) {
#pragma unroll
                    for (u32 t = 0; t < PN_B_BYTES / 16 / 32; t++) bv[V ? 0 : t] = __ldg(bsrc + lane + 32 * t);
                }
                const u32 nw = ((mt_pack >> (4 * k)) & 15u) * 4;
                const u32 sgq = Q / PN_SUB, slot = sgq % PN_NSTG, sub = Q % PN_NSTAGES;  // stage, its ring slot, my sub-slot (= slot * 4 + ks)
                if (sgq >= PN_NSTG) mbar_wait(empty0 + 8 * slot, (sgq / PN_NSTG - 1) & 1u);
                const u32 st = sS_addr + sub * PN_STAGE_BYTES;
                if (V == 1 && lane == 0) {  // the slot is free: start the bulk copy of the digit rows, its bytes complete on the stage's barrier
                    mbar_expect_tx(full0 + 8 * slot, PN_B_BYTES);
                    bulk_g2s(st + PN_A_BYTES, bsrc, PN_B_BYTES, full0 + 8 * slot);
                }
#pragma unroll
                for (u32 j = 0; j < 12; j++) {
                    if (j < nw) {
                        uint4 lo, hi;
                        expand_bits32(cur[j], lo, hi);
                        const u32 a0 = st + (j >> 2) * 4096 + (2 * (j & 3)) * 512 + lane * 16;
                        st_shared_v4(a0, lo);
                        st_shared_v4(a0 + 512, hi);
                    }
                }
                if (V == 0) {
#pragma unroll
                    for (u32 t = 0; t < PN_B_BYTES / 16 / 32; t++) st_shared_v4(st + PN_A_BYTES + (lane + 32 * t) * 16, bv[V ? 0 : t]);
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(full0 + 8 * slot);
                Q += PW;
                tile = ntile;
                r = nr;
                ks = nks;
                k = nk;
                live = more;
                if (more) {
#pragma unroll
                    for (u32 j = 0; j < 12; j++) cur[j] = nxt[j];
                }
            }
        }
        Q0 += (u32)(t_end - t_begin) * PN_SUB * nlev;
        fence_before_sync();
        __syncthreads();  // item boundary: the epilogue has read the accumulators, every stage was consumed, next item id visible
        fence_after_sync();
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc_512(tmem);
}

// ---------------------------------------------------------------- launchers
static int scales_from_colmax(sb_ctx *ctx, DevBuf<unsigned long long> &colmax, DevBuf<double> &scale2, DevBuf<int> &ex) {
    SB_TRY(scale2.ensure(PL_COLS));
    SB_TRY(ex.ensure(PL_COLS));
    k_pl_scales<<<1, 32, 0, ctx->stream>>>(colmax.p, scale2.p, ex.p);
    count_launch(ctx);
    return SB_OK;
}

// gather.cu
int gather_run_tile(sb_ctx *ctx, const GatherLayout &L, int mode, const MapDev &mp, u64 n_cells, const double *B, u32 ldb, u32 w, u32 col0, double *out,
                    u32 ldo, long long *cycles);

// T[c, :] += the plane part of A^T . Y   (out already holds the offset term; the sparse gather adds the rest).
// With `gl` (log chain): the sparse gather over that layout is run here as well, per column pass, with its run factor L_c(1)
// deferred -- its sums land in one more block behind the per-unit partial rows and k_pl_reduce_t folds l1[c] * block into T.
int planes_t(sb_nmat *a, const double *Y, u32 ldy, u32 w, double *out, u32 ldo, const GatherLayout *gl, const MapDev *mp, long long *cycles) {
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    const PlaneSet &pl = mt->pl;
    if (!pl.active || mt->n == 0 || w == 0) return SB_OK;
    const u32 G1 = pl.G[0];
    const u32 nranges = (G1 + PT_RANGE - 1) / PT_RANGE;
    const u64 n_pad = pl.ntiles * PL_TILE;
    DevBuf<unsigned long long> &colmax = pl.ws_colmax;
    DevBuf<signed char> &Bd = pl.ws_bd;
    DevBuf<double> &scale2 = pl.ws_scale2, &part = pl.ws_part;
    DevBuf<int> &ex = pl.ws_ex;
    SB_TRY(colmax.ensure(PL_COLS));
    SB_TRY(Bd.ensure((size_t)nranges * PT_B_BYTES));
    SB_TRY(part.ensure((size_t)(pl.n_units_t + (gl ? 1 : 0)) * n_pad * PL_COLS));
    double *t1 = gl ? part.p + (size_t)pl.n_units_t * n_pad * PL_COLS : nullptr;
    const double *rs = a->has_row_scale ? a->row_scale.p : nullptr;
    const size_t smem = (size_t)PT_B_BYTES + PT_NSTAGES * PT_STAGE_BYTES + sizeof(PtShared);
    const bool v1 = ctx->pl_variant & 1;
    cudaError_t e = v1 ? cudaFuncSetAttribute(k_planes_t<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                       : cudaFuncSetAttribute(k_planes_t<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return sb_fail(SB_ERR_CUDA, "planes_t: %zu B of shared memory: %s", smem, cudaGetErrorString(e));
    const u32 items = G1 * PL_COLS;
    const unsigned rblocks = (unsigned)std::max<u64>(1, std::min<u64>((mt->n * (PL_COLS / 2) + 255) / 256, (u64)ctx->sm_count * 16));
    for (u32 col0 = 0; col0 < w; col0 += PL_COLS) {
        const u32 wt = std::min(PL_COLS, w - col0);
        SB_CUDA(cudaMemsetAsync(colmax.p, 0, PL_COLS * sizeof(unsigned long long), ctx->stream));
        if (col0 == 0) SB_CUDA(cudaMemsetAsync(Bd.p, 0, (size_t)nranges * PT_B_BYTES, ctx->stream));  // padding columns / ranks stay zero
        k_pl_colmax_t<<<cdiv(items, 256), 256, 0, ctx->stream>>>(Y, ldy, mt->hot_idx.p, rs, G1, col0, wt, colmax.p);
        SB_TRY(scales_from_colmax(ctx, colmax, scale2, ex));
        k_pl_digits_t<<<cdiv(items, 256), 256, 0, ctx->stream>>>(Y, ldy, mt->hot_idx.p, rs, G1, col0, wt, ex.p, Bd.p, v1 ? 1u : 0u);
        SB_CUDA(cudaMemsetAsync(pl.counter.p, 0, sizeof(u32), ctx->stream));
        if (gl) {  // the sparse half of this column pass, in units of L_c(1)
            SB_CUDA(cudaMemsetAsync(t1, 0, (size_t)mt->n * PL_COLS * sizeof(double), ctx->stream));
            SB_TRY(gather_run_tile(ctx, *gl, 2, *mp, mt->n, Y, ldy, w, col0, t1 - col0, PL_COLS, col0 == 0 ? cycles : nullptr));
        }
        if (v1)
            k_planes_t<1><<<pl.t_grid, PtLayout<1>::WARPS * 32, smem, ctx->stream>>>(make_pldev(mt), (const PlUnitT *)pl.units_t.p,
                                                                                     (const PlItem *)pl.items_t.p, pl.n_items_t, pl.counter.p, Bd.p, scale2.p,
                                                                                     a->lk.p, wt, part.p, (u32)ctx->pl_debug);
        else
            k_planes_t<0><<<pl.t_grid, PtLayout<0>::WARPS * 32, smem, ctx->stream>>>(make_pldev(mt), (const PlUnitT *)pl.units_t.p,
                                                                                     (const PlItem *)pl.items_t.p, pl.n_items_t, pl.counter.p, Bd.p, scale2.p,
                                                                                     a->lk.p, wt, part.p, (u32)ctx->pl_debug);
        k_pl_reduce_t<<<rblocks, 256, 0, ctx->stream>>>(part.p, pl.n_units_t, mt->n, n_pad, col0, wt, out, ldo, t1, gl ? a->l1c.p : nullptr);
        count_launch(ctx); count_launch(ctx); count_launch(ctx); count_launch(ctx);
    }
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

static int planes_n_impl(sb_nmat *a, const double *X, u32 ldx, u32 w, int mode, double *out, u64 row_stride, u64 col_stride) {
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    const PlaneSet &pl = mt->pl;
    if (!pl.active || mt->n == 0 || w == 0) return SB_OK;
    const u64 n_pad = pl.ntiles * PL_TILE;
    DevBuf<unsigned long long> &colmax = pl.ws_colmax;
    DevBuf<signed char> &Bn = pl.ws_bn;
    DevBuf<double> &scale2 = pl.ws_scale2;
    DevBuf<int> &ex = pl.ws_ex;
    SB_TRY(colmax.ensure(PL_COLS));
    SB_TRY(Bn.ensure((size_t)pl.L * (n_pad / 8) * PN_CELLGRP_BYTES));
    const size_t smem = (size_t)PN_NSTAGES * PN_STAGE_BYTES + sizeof(PnShared);
    const bool v1 = ctx->pl_variant & 2;
    cudaError_t e = v1 ? cudaFuncSetAttribute(k_planes_n<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                       : cudaFuncSetAttribute(k_planes_n<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return sb_fail(SB_ERR_CUDA, "planes_n: %zu B of shared memory: %s", smem, cudaGetErrorString(e));
    const int cm_blocks = (int)std::max<u64>(1, std::min<u64>((mt->n + 255) / 256, (u64)ctx->sm_count * 4));
    for (u32 col0 = 0; col0 < w; col0 += PL_COLS) {
        const u32 wt = std::min(PL_COLS, w - col0);
        SB_CUDA(cudaMemsetAsync(colmax.p, 0, PL_COLS * sizeof(unsigned long long), ctx->stream));
        k_pl_colmax_n<<<cm_blocks, 256, 0, ctx->stream>>>(X, ldx, mt->n, a->lk.p, pl.L, col0, wt, mode, colmax.p);
        SB_TRY(scales_from_colmax(ctx, colmax, scale2, ex));
        k_pl_digits_n<<<cdiv(n_pad * pl.L, 128), 128, 0, ctx->stream>>>(X, ldx, mt->n, n_pad, a->lk.p, pl.L, col0, wt, mode, ex.p, Bn.p);
        SB_CUDA(cudaMemsetAsync(pl.counter.p, 0, sizeof(u32), ctx->stream));
        if (v1)
            k_planes_n<1><<<pl.n_grid, (PL_EPI_WARPS + 1 + 12) * 32, smem, ctx->stream>>>(make_pldev(mt), (const PlUnitN *)pl.units_n.p,
                                                                                          (const PlItem *)pl.items_n.p, pl.n_items_n, pl.counter.p, Bn.p, n_pad,
                                                                                          scale2.p, mt->hot_idx.p, col0, wt, out, row_stride, col_stride);
        else
            k_planes_n<0><<<pl.n_grid, PL_THREADS, smem, ctx->stream>>>(make_pldev(mt), (const PlUnitN *)pl.units_n.p, (const PlItem *)pl.items_n.p,
                                                                        pl.n_items_n, pl.counter.p, Bn.p, n_pad, scale2.p, mt->hot_idx.p, col0, wt, out,
                                                                        row_stride, col_stride);
        count_launch(ctx); count_launch(ctx); count_launch(ctx);
    }
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

// P[g, :] += the plane part of sum_c L_c(v_gc) X[c, :]   (row scale and offset are applied by k_spmm_n_finalize)
int planes_n(sb_nmat *a, const double *X, u32 ldx, u32 w, double *P, u32 ldp) { return planes_n_impl(a, X, ldx, w, 0, P, ldp, 1); }

// S1[g] += sum_c L, S2[g] += sum_c L^2 over the plane entries
int planes_moments(sb_nmat *a, double *S1, double *S2) {
    if (S2 < S1) return sb_fail(SB_ERR_UNSUPPORTED, "planes_moments: S2 must follow S1");
    return planes_n_impl(a, nullptr, 0, 2, 1, S1, 1, (u64)(S2 - S1));
}
