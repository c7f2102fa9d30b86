// gather.cu -- the panelled sparse gather behind both products of the Krylov loop (the cold half of the
// hybrid layout, or every entry when a matrix has no planes).
//
//   N side (K8)  P[g,:] += sum_c x_gc * X[c,:]      restates low_rank_offset.rs:68-81 -> mat.rs:1074-1090 -> prod.rs:30-51,87-148
//       stream: cell panels of `rows` cells, inside a panel sorted by (gene, cell); entry {gene | cell_local << 22, count}
//   T side (K7)  T[c,:] += sum_g x_gc * Y[g,:]      restates low_rank_offset.rs:83-96 -> mat.rs:1114-1133 -> prod.rs:56-81,154-214
//       stream: blocks of GA_TBLOCK cells; inside a block gene panels of `rows` gene slots (genes ranked by how many
//       cells express them); inside a (block, panel) sorted by (cell, gene); entry {cell | slot_local << 22, count}
//
// One kernel serves both: the panel's rows of the dense block (X rows of the panel's cells, or row-scaled Y rows of the
// panel's genes) are staged in shared memory once per work unit, and the stream is a sequence of *runs* of one output
// row (gene on the N side, cell on the T side).  Why this shape (ncu, DESIGN.md 3): a width-20 f64 gather moves 160 B of
// operand per 8-byte entry, so the kernel lives or dies by shared-memory wavefronts and by how often a run's partial
// row has to be flushed to memory.
//   * Operand rows are split into a 128-byte part (columns 0..15) and a 32-byte tail (16..19).  A group of 8 lanes
//     covers the 128-byte part with one LDS.128 per lane = exactly one conflict-free wavefront per entry (a 160-byte row
//     read by 10 lanes straddles the quarter-warp phases and costs ~1.8).  The tails of two consecutive entries share
//     one LDS.64.
//   * Each 8-lane group walks its OWN contiguous span of the stream, so a run's partial sums live in one group's
//     registers: a flush is 20 f64 reductions (RED.ADD.F64), not 20 per lane group, and needs no cross-group shuffles.
//   * The entry scalars {map value, row offset, run key, head flag} are computed once by the lane that loaded the entry
//     and handed to the group through a padded per-group staging buffer (one broadcast LDS.128 per step).
// The normalization map is evaluated in the load (the normalized matrix is never materialised).
#include <cub/cub.cuh>

#include <algorithm>
#include <numeric>

#include "common.cuh"
#include "map.cuh"

#define FULLMASK 0xffffffffu
#define GA_THREADS 1024
#define GA_STAGE_STRIDE 176u  // bytes per 8-lane group in the staging buffer (44 words: neighbouring groups land in different banks)
#define GA_NONE 0xFFFFFFFFu
#define GA_TILE 20u           // columns per pass: 16 (main) + 4 (tail)

// ---------------------------------------------------------------- the kernel
// Staging buffer of one 8-lane group (GA_STAGE_STRIDE bytes): offs[8] u16 (row offset / 16) | keys[8] u32 | xs[8] f64 | l1s[8] f64
#define GA_ST_KEYS 16u
#define GA_ST_XS 48u
#define GA_ST_L1 112u

// MODE 0: N side, 1: T side, 2: T side with the run factor deferred -- the sums of a cell's runs leave in units of L_c(1) (`out` is
// then a separate block that the caller scales by L_c(1) and adds to T: k_pl_reduce_t), so the kernel loads no per-cell factor at
// the run heads (ncu: 28 % of the T side's stall samples sat on those global loads) and multiplies nothing at the flush.
// TAIL: the pass has columns 16..19
template <int MODE, int TAIL>
__global__ void __launch_bounds__(GA_THREADS, 1)
k_gather(const uint2 *__restrict__ ent, const GUnit *__restrict__ units, const u32 *__restrict__ item_first, u32 n_units, u32 n_items,
         u32 *__restrict__ tickets, u32 ticket_base, u32 rows, u64 n_cells, MapDev mp, const double *__restrict__ B, u32 ldb, u32 col0, u32 wt, u32 w,
         const u32 *__restrict__ slot_gene, double *__restrict__ out, u32 ldo, long long *__restrict__ cycles) {
    __shared__ u32 s_item;
    __shared__ long long s_t0;
    if (cycles && threadIdx.x == 0) s_t0 = clock64();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *XA = reinterpret_cast<double *>(smem_raw);                   // (rows + 1) x 16; row `rows` is all zero
    double *XB = XA + (size_t)(rows + 1) * 16;                            // (rows + 1) x 4 (TAIL only)
    double *par = XB + (TAIL ? (size_t)(rows + 1) * 4 : 0);               // rows: N: column parameter of the cell; T: binomial pi of the gene
    double *par2 = par + rows;                                            // rows: N, log chain: 1 / L_c(1)
    LogEnt *ltab = reinterpret_cast<LogEnt *>(par2 + rows);               // 128 (rows is even: 16-byte aligned)
    unsigned char *stage_all = reinterpret_cast<unsigned char *>(ltab + 128);

    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int grp = lane >> 3, lig = lane & 7;
    const u32 xa_sa = (u32)__cvta_generic_to_shared(XA) + (u32)lig * 16u;
    const u32 xb_sa = (u32)__cvta_generic_to_shared(XB) + (u32)(lig & 3) * 8u;
    const u32 stage_grp = (u32)__cvta_generic_to_shared(stage_all) + (u32)(wib * 4 + grp) * GA_STAGE_STRIDE;
    const u32 zero_off16 = rows * 8u;  // row offsets travel as bytes / 16 in a u16
    const u32 cA = 2u * lig, cB = 16u + (lig & 3);
    const bool ok0 = cA < wt && col0 + cA < w, ok1 = cA + 1 < wt && col0 + cA + 1 < w;
    const bool okb = TAIL && cB < wt && col0 + cB < w;
    const u32 wt_even = (wt + 1) & ~1u;
    const bool logchain = mp.kind == 1;
    constexpr bool TS = MODE >= 1, DEFER = MODE == 2;
    double *const oA = out + col0 + cA;
    const long long tdelta = (long long)cB - (long long)cA;  // tail column relative to this lane's first main column
    const u32 ok0m = ok0, ok1m = ok1, okbm = okb;
    const u64 ldo64 = (u64)ldo;

    for (int i = threadIdx.x; i < 128; i += blockDim.x) ltab[i] = sb_log_table[i];

    u32 staged = GA_NONE;
    u32 first_item = GA_NONE;  // calibration pass (one item per CTA): the share this CTA drew

    // Persistent CTAs draw work items (runs of units, panel-major) from a ticket counter: the cost model that cuts the T-side line
    // into items is only approximate (ncu: sm__cycles_active 1.19 / 1.49 / 1.79 M min / avg / max with one static share per CTA),
    // so the line is cut several times finer than the grid and whoever finishes early takes the next piece -- usually of the
    // panel it has already staged.
    for (;;) {
    __syncthreads();  // every warp is done with the previous item (and has read s_item)
    if (threadIdx.x == 0) s_item = atomicAdd(tickets, 1u) - ticket_base;
    __syncthreads();
    const u32 item = s_item;
    if (item >= n_items) break;
    if (first_item == GA_NONE) first_item = item;
    const u32 u_begin = item_first[item], u_end = min(n_units, item_first[item + 1]);
    for (u32 ui = u_begin; ui < u_end; ui++) {
        const GUnit un = units[ui];
        if (un.panel != staged) {
            __syncthreads();  // readers of the previous panel are done
            constexpr u32 PAIRS = TAIL ? 10 : 8;
            for (u32 i = threadIdx.x; i < (rows + 1) * PAIRS; i += blockDim.x) {
                const u32 r = i / PAIRS, j2 = (i - r * PAIRS) * 2, col = col0 + j2;
                double2 val = make_double2(0.0, 0.0);
                if (r < rows && j2 < wt_even && col < w) {  // ldb and col are even, so col < w <= ldb implies col + 1 < ldb
                    if (MODE == 0) {
                        // log chain: the row of cell c is staged as L_c(1) . X[c,:], so an entry with count 1 is a plain add
                        const u64 cell = (u64)un.panel * rows + r;
                        if (cell < n_cells) {
                            val = *reinterpret_cast<const double2 *>(B + cell * (size_t)ldb + col);
                            if (logchain) {
                                const double l1 = mp.l1[cell];
                                val.x *= l1;
                                val.y *= l1;
                            }
                        }
                    } else {
                        const u32 g = slot_gene[(size_t)un.panel * rows + r];
                        if (g != GA_NONE) {
                            val = *reinterpret_cast<const double2 *>(B + (size_t)g * ldb + col);
                            if (logchain && mp.row) {  // the row scale of the log chain rides on the staged rows
                                const double rs = mp.row[g];
                                val.x *= rs;
                                val.y *= rs;
                            }
                        }
                    }
                }
                if (j2 < 16) *reinterpret_cast<double2 *>(XA + (size_t)r * 16 + j2) = val;
                else *reinterpret_cast<double2 *>(XB + (size_t)r * 4 + (j2 - 16)) = val;
            }
            for (u32 r = threadIdx.x; r < rows; r += blockDim.x) {
                double pv = 0.0, pv2 = 0.0;
                if (MODE == 0) {
                    const u64 cell = (u64)un.panel * rows + r;
                    if (cell < n_cells) {
                        pv = mp.col[cell];
                        if (logchain) pv2 = mp.inv_l1[cell];
                    }
                } else if (!logchain) {
                    const u32 g = slot_gene[(size_t)un.panel * rows + r];
                    if (g != GA_NONE) pv = mp.row[g];
                }
                par[r] = pv;
                par2[r] = pv2;
            }
            staged = un.panel;
            __syncthreads();
        }
        // warp span (multiple of 32 entries), cut into four group spans (multiples of 8)
        u64 span = (un.end - un.begin + nw - 1) / nw;
        span = (span + 31) & ~(u64)31;
        const u64 wb = min(un.end, un.begin + (u64)wib * span), we = min(un.end, wb + span);
        const u64 qspan = span >> 2;
        const u64 gb = min(we, wb + (u64)grp * qspan), ge = min(we, gb + qspan);
        const u32 nchunks = (u32)((min(we, wb + qspan) - wb + 7) >> 3);  // group 0 has the longest span

        // cur: output row of the run in flight; uniform inside a group
        u32 cur = GA_NONE, carry = GA_NONE;
        double curL1 = 0.0;  // T side: L_cur(1), applied to the run's sum at the flush
        double a0 = 0.0, a1 = 0.0, bt = 0.0;

        auto flush = [&]() {
            if (cur == GA_NONE) return;  // nothing accumulated yet (and never reduce zeros into one shared row)
            if (TS && !DEFER) {
                a0 *= curL1;
                a1 *= curL1;
                bt *= curL1;
            }
            // three predicated f64 reductions off one address computation
            double *o = oA + (u64)cur * ldo64;
            asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p red.global.add.f64 [%0], %1; }" ::"l"(o), "d"(a0), "r"(ok0m) : "memory");
            asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p red.global.add.f64 [%0 + 8], %1; }" ::"l"(o), "d"(a1), "r"(ok1m) : "memory");
            if (TAIL) asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p red.global.add.f64 [%0], %1; }" ::"l"(o + tdelta), "d"(bt), "r"(okbm) : "memory");
            a0 = 0.0;
            a1 = 0.0;
            bt = 0.0;
        };

        uint2 znext = (gb + lig < ge) ? __ldcs(ent + gb + lig) : make_uint2(GA_NONE, 0u);
        for (u32 ch = 0; ch < nchunks; ch++) {
            const uint2 z = znext;
            const u64 kn = gb + (u64)(ch + 1) * 8 + lig;
            znext = (kn < ge) ? __ldcs(ent + kn) : make_uint2(GA_NONE, 0u);
            const bool valid = z.x != GA_NONE;
            const u32 key = z.x & SB_GENE_MASK, local = z.x >> SB_GENE_BITS;
            // general entries carry an explicit factor; a count of 1 under the log chain is the staged row itself (N side)
            // or is scaled once per run at the flush (T side)
            const bool general = valid && (!logchain || z.y != 1u);
            double x = 0.0;
            if (general) {
                if (MODE == 0) {
                    if (logchain) x = map_log_part(mp.log_base, par[local], z.y, ltab) * par2[local];
                    else x = map_full(mp, z.y, key, par[local], false, ltab);
                } else {
                    const double cp = mp.col[key];
                    if (logchain) x = map_log_part(mp.log_base, cp, z.y, ltab) * mp.inv_l1[key];
                    else x = mp.kind == 2 ? map_binom_dev((double)z.y, cp, par[local]) : map_binom_pearson((double)z.y, cp, par[local]);
                }
            }
            u32 prev = __shfl_up_sync(FULLMASK, key, 1, 8);
            if (lig == 0) prev = carry;
            const bool head = valid && key != prev;
            // T side: L_c(1) is consumed once per run (at its flush): only the entry that opens a run fetches it
            double l1v = 0.0;
            if (TS && !DEFER && head) l1v = logchain ? mp.l1[key] : 1.0;
            carry = __shfl_sync(FULLMASK, key, 7, 8);
            const u32 myh = (__ballot_sync(FULLMASK, head) >> (8 * grp)) & 0xFFu;
            const u32 myg = (__ballot_sync(FULLMASK, general) >> (8 * grp)) & 0xFFu;
            __syncwarp();
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(stage_grp + (u32)lig * 2u), "h"((unsigned short)(valid ? local * 8u : zero_off16)) : "memory");
            asm volatile("st.shared.u32 [%0], %1;" ::"r"(stage_grp + GA_ST_KEYS + (u32)lig * 4u), "r"(key) : "memory");
            if (general) asm volatile("st.shared.f64 [%0], %1;" ::"r"(stage_grp + GA_ST_XS + (u32)lig * 8u), "d"(x) : "memory");
            if (TS && !DEFER && head) asm volatile("st.shared.f64 [%0], %1;" ::"r"(stage_grp + GA_ST_L1 + (u32)lig * 8u), "d"(l1v) : "memory");
            __syncwarp();
            u32 ov[4];
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(ov[0]), "=r"(ov[1]), "=r"(ov[2]), "=r"(ov[3]) : "r"(stage_grp));
#pragma unroll
            for (int s = 0; s < 8; s += 2) {
                const u32 off0 = (ov[s >> 1] & 0xFFFFu) << 4, off1 = (ov[s >> 1] >> 16) << 4;
                double tl = 0.0;
                if (TAIL) {  // lanes 0..3 take the tail of entry s, lanes 4..7 the tail of entry s + 1: one LDS.64 for both
                    const u32 toff = (lig < 4 ? off0 : off1) >> 2;
                    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(tl) : "r"(xb_sa + toff));
                }
                double x0, x1, m0 = 1.0, m1 = 1.0;
                asm volatile("{ .reg .pred p; setp.ne.u32 p, %1, 0; @p ld.shared.f64 %0, [%2]; }"
                             : "+d"(m0) : "r"(myg & (1u << s)), "r"(stage_grp + GA_ST_XS + (u32)s * 8u));
                asm volatile("{ .reg .pred p; setp.ne.u32 p, %1, 0; @p ld.shared.f64 %0, [%2]; }"
                             : "+d"(m1) : "r"(myg & (2u << s)), "r"(stage_grp + GA_ST_XS + (u32)(s + 1) * 8u));
                if (myh & (1u << s)) {
                    flush();
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(cur) : "r"(stage_grp + GA_ST_KEYS + (u32)s * 4u));
                    if (TS && !DEFER) asm volatile("ld.shared.f64 %0, [%1];" : "=d"(curL1) : "r"(stage_grp + GA_ST_L1 + (u32)s * 8u));
                }
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x0), "=d"(x1) : "r"(xa_sa + off0));
                a0 = fma(m0, x0, a0);
                a1 = fma(m0, x1, a1);
                if (TAIL && lig < 4) bt = fma(m0, tl, bt);
                if (myh & (2u << s)) {
                    flush();
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(cur) : "r"(stage_grp + GA_ST_KEYS + (u32)(s + 1) * 4u));
                    if (TS && !DEFER) asm volatile("ld.shared.f64 %0, [%1];" : "=d"(curL1) : "r"(stage_grp + GA_ST_L1 + (u32)(s + 1) * 8u));
                }
                asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x0), "=d"(x1) : "r"(xa_sa + off1));
                a0 = fma(m1, x0, a0);
                a1 = fma(m1, x1, a1);
                if (TAIL && lig >= 4) bt = fma(m1, tl, bt);
            }
        }
        flush();
    }
    }
    if (cycles && threadIdx.x == 0 && first_item != GA_NONE) {  // busy time of the share's CTA and the SM it ran on (calibration pass only)
        u32 smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        cycles[first_item] = clock64() - s_t0;
        cycles[gridDim.x + first_item] = (long long)smid;
    }
}

// out[c, j] = v_c * uy[j] (or 0): the rank-1 offset of A^T.Y; the plane kernels and the gather add on top
__global__ void k_t_init(double *__restrict__ out, u64 n, u32 w, u32 ldo, const double *__restrict__ uy, const double *__restrict__ v) {
    const u64 total = n * w;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (u64)gridDim.x * blockDim.x) {
        const u64 c = i / w;
        const u32 j = (u32)(i - c * w);
        out[c * ldo + j] = uy ? (v ? v[c] : 1.0) * uy[j] : 0.0;
    }
}

int gather_t_init(sb_ctx *ctx, double *out, u64 n, u32 w, u32 ldo, const double *uy, const double *v) {
    if (n == 0 || w == 0) return SB_OK;
    u64 blocks = std::min<u64>((n * w + 255) / 256, (u64)ctx->sm_count * 16);
    k_t_init<<<(unsigned)blocks, 256, 0, ctx->stream>>>(out, n, w, ldo, uy, v);
    count_launch(ctx);
    return SB_OK;
}

static size_t gather_smem(u32 rows, bool tail) {
    return (size_t)(rows + 1) * (tail ? 20 : 16) * 8 + (size_t)rows * 16 + 128 * sizeof(LogEnt) + (size_t)(GA_THREADS / 32) * 4 * GA_STAGE_STRIDE;
}

// one column pass (columns [col0, col0 + min(20, w - col0))) of one product over a layout.  mode 0: N side; 1: T side; 2: T side with
// the run factor L_c(1) deferred to the caller (`out` + col0 then addresses a separate block, see k_gather)
int gather_run_tile(sb_ctx *ctx, const GatherLayout &L, int mode, const MapDev &mp, u64 n_cells, const double *B, u32 ldb, u32 w, u32 col0, double *out,
                    u32 ldo, long long *cycles) {
    if (!L.ready) return sb_fail(SB_ERR_UNSUPPORTED, "gather_run: layout not built");
    if (L.nnz == 0 || L.n_units == 0 || w == 0 || col0 >= w) return SB_OK;
    const u32 n_items = L.n_items ? L.n_items : L.grid;
    if (!L.tickets.p) {
        SB_TRY(L.tickets.alloc(1));
        SB_CUDA(cudaMemsetAsync(L.tickets.p, 0, sizeof(u32), ctx->stream));
        L.ticket_base = 0;
    }
    if (L.ticket_base > 0x7F000000u) {  // long before the u32 ticket counter could wrap
        SB_CUDA(cudaMemsetAsync(L.tickets.p, 0, sizeof(u32), ctx->stream));
        L.ticket_base = 0;
    }
    const u32 wt = std::min(GA_TILE, w - col0);
    const bool tail = wt > 16;
    const size_t smem = gather_smem(L.rows, tail);
    cudaError_t e;
#define GA_LAUNCH(M, T)                                                                                                                        \
    e = cudaFuncSetAttribute(k_gather<M, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                                          \
    if (e == cudaSuccess)                                                                                                                      \
        k_gather<M, T><<<L.grid, GA_THREADS, smem, ctx->stream>>>(L.ent, L.units.p, L.cta_first.p, L.n_units, n_items, L.tickets.p, L.ticket_base, \
                                                                  L.rows, n_cells, mp, B, ldb, col0, wt, w, L.slot_gene.p, out, ldo, cycles);
    if (mode == 0) {
        if (tail) { GA_LAUNCH(0, 1) } else { GA_LAUNCH(0, 0) }
    } else if (mode == 1) {
        if (tail) { GA_LAUNCH(1, 1) } else { GA_LAUNCH(1, 0) }
    } else {
        if (tail) { GA_LAUNCH(2, 1) } else { GA_LAUNCH(2, 0) }
    }
#undef GA_LAUNCH
    if (e != cudaSuccess) return sb_fail(SB_ERR_CUDA, "gather_run: %zu B of shared memory: %s", smem, cudaGetErrorString(e));
    L.ticket_base += n_items + L.grid;
    count_launch(ctx);
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

// runs all column passes of one product over a layout
int gather_run(sb_ctx *ctx, const GatherLayout &L, int mode, const MapDev &mp, u64 n_cells, const double *B, u32 ldb, u32 w, double *out, u32 ldo,
               long long *cycles) {
    for (u32 col0 = 0; col0 < w; col0 += GA_TILE) SB_TRY(gather_run_tile(ctx, L, mode, mp, n_cells, B, ldb, w, col0, out, ldo, col0 == 0 ? cycles : nullptr));
    return SB_OK;
}

// ---------------------------------------------------------------- N-side units: equal nnz per CTA, cut at panel boundaries
int gather_build_n(sb_mat *mt, GatherLayout &L, const uint2 *gm, const u64 *gm_base_dev, u64 nnz) {
    sb_ctx *ctx = mt->ctx;
    L.ready = false;
    L.rows = (mt->pc + 1) & ~1u;
    if (L.rows != mt->pc) return sb_fail(SB_ERR_UNSUPPORTED, "gather_build_n: odd panel size");
    L.npanels = mt->np;
    L.ent = gm;
    L.nnz = nnz;
    std::vector<u64> base((size_t)mt->np + 1, 0);
    if (mt->np) SB_CUDA(cudaMemcpyAsync(base.data(), gm_base_dev, base.size() * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    const u32 G = (u32)ctx->sm_count;
    std::vector<GUnit> units;
    std::vector<u32> first;
    gather_units_n(base, nnz, G, units, first);
    L.n_units = (u32)units.size();
    L.grid = G;
    SB_TRY(L.units.alloc(units.size()));
    SB_TRY(L.cta_first.alloc(first.size()));
    if (!units.empty()) SB_CUDA(cudaMemcpyAsync(L.units.p, units.data(), units.size() * sizeof(GUnit), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(L.cta_first.p, first.data(), first.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    L.ready = true;
    return SB_OK;
}

// ---------------------------------------------------------------- T-side layout
__global__ void k_ent_gene_hist(const uint2 *__restrict__ ent, u64 nnz, u32 *__restrict__ hist) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (u64)gridDim.x * blockDim.x) atomicAdd(&hist[ent[i].x], 1u);
}

// one warp per cell of the range: key = (cell block inside the range) * npanels + gene panel, payload = packed T-side entry
__global__ void k_make_tkeys(const u64 *__restrict__ ptr, const uint2 *__restrict__ ent, u64 nc, u64 c0, const u32 *__restrict__ slot_of_gene,
                             u32 rows, u32 npanels, u32 *__restrict__ keys, u64 *__restrict__ payload) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 v = warp; v < nc; v += nwarps) {
        const u64 s = ptr[v], e = ptr[v + 1];
        const u32 blk = (u32)(v / GA_TBLOCK);
        const u32 cell = (u32)(c0 + v);
        for (u64 k = s + lane; k < e; k += 32) {
            const uint2 z = ent[k];
            const u32 slot = slot_of_gene[z.x];
            const u32 p = slot / rows, sl = slot - p * rows;
            keys[k] = blk * npanels + p;
            payload[k] = ((u64)z.y << 32) | (u64)(cell | (sl << SB_GENE_BITS));
        }
    }
}

__global__ void k_unpack_u64(const u64 *__restrict__ payload, uint2 *__restrict__ out, u64 nnz) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (u64)gridDim.x * blockDim.x) {
        const u64 p = payload[i];
        out[i] = make_uint2((u32)p, (u32)(p >> 32));
    }
}

// first[key] = first entry of a (block, panel) segment; runs[key] = number of runs (distinct cells) inside it
__global__ void k_key_first(const u32 *__restrict__ keys, const u64 *__restrict__ payload, u64 nnz, u64 *__restrict__ first,
                            unsigned long long *__restrict__ runs) {
    const int lane = threadIdx.x & 31;
    const u64 total = (nnz + 31) & ~(u64)31;  // whole warps stay in the loop together
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (u64)gridDim.x * blockDim.x) {
        const bool valid = i < nnz;
        const u32 key = valid ? keys[i] : 0xFFFFFFFFu;
        bool head = false;
        if (valid) {
            const bool newkey = i == 0 || keys[i - 1] != key;
            if (newkey) first[key] = i;
            head = newkey || ((u32)payload[i - 1] & SB_GENE_MASK) != ((u32)payload[i] & SB_GENE_MASK);
        }
        const u32 key0 = __shfl_sync(FULLMASK, key, 0);
        const unsigned hm = __ballot_sync(FULLMASK, head);
        if (__all_sync(FULLMASK, !valid || key == key0)) {
            if (lane == 0 && hm) atomicAdd(&runs[key0], (unsigned long long)__popc(hm));
        } else if (head) {
            atomicAdd(&runs[key], 1ull);
        }
    }
}

static inline int ga_grid(u64 items, int threads, sb_ctx *ctx, int per_sm = 16) {
    u64 blocks = (items + threads - 1) / threads, cap = (u64)ctx->sm_count * per_sm;
    return (int)std::max<u64>(1, std::min(blocks, cap));
}

// ranks the genes by how many entries of the sample they have and assigns gene slots (rank -> panel, row)
int gather_assign_slots(sb_mat *mt, const uint2 *ent, u64 nnz) {
    sb_ctx *ctx = mt->ctx;
    GatherLayout &L = mt->gt;
    L.ready = false;
    const u32 m = mt->m;
    u32 rows = std::min<u32>(SB_MAX_PANEL_CELLS, (m + 1) & ~1u);
    if (rows < 2) rows = 2;
    L.rows = rows;
    L.npanels = (m + rows - 1) / rows;
    if (L.npanels == 0) L.npanels = 1;
    DevBuf<u32> hist;
    SB_TRY(hist.alloc((size_t)m + 1));
    SB_CUDA(cudaMemsetAsync(hist.p, 0, ((size_t)m + 1) * sizeof(u32), ctx->stream));
    if (nnz) {
        k_ent_gene_hist<<<ga_grid(nnz, 256, ctx), 256, 0, ctx->stream>>>(ent, nnz, hist.p);
        count_launch(ctx);
    }
    std::vector<u32> h((size_t)m + 1);
    SB_CUDA(cudaMemcpyAsync(h.data(), hist.p, h.size() * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    std::vector<u32> order(m);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](u32 a, u32 b) { return h[a] > h[b]; });
    std::vector<u32> slot_of(m ? m : 1, 0), slot_gene((size_t)L.npanels * rows, GA_NONE);
    for (u32 r = 0; r < m; r++) {
        slot_of[order[r]] = r;
        slot_gene[r] = order[r];
    }
    SB_TRY(mt->slot_of_gene.alloc(slot_of.size()));
    SB_TRY(L.slot_gene.alloc(slot_gene.size()));
    SB_CUDA(cudaMemcpyAsync(mt->slot_of_gene.p, slot_of.data(), slot_of.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(L.slot_gene.p, slot_gene.data(), slot_gene.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// T-side order of the cells [c0, c0 + nc) (c0 a multiple of GA_TBLOCK) given their range-local cell-major pair.
// seg_len receives the entry count of every (block, panel) of the range, in stream order.
int gather_build_t_range(sb_mat *mt, u64 c0, u64 nc, const u64 *ptr_local, const uint2 *ent, u64 nnz, DevBuf<uint2> &out, std::vector<u64> &seg_len,
                         std::vector<u64> &seg_runs) {
    sb_ctx *ctx = mt->ctx;
    GatherLayout &L = mt->gt;
    const u64 nblk = (nc + GA_TBLOCK - 1) / GA_TBLOCK;
    const u64 nkeys = nblk * L.npanels;
    seg_len.assign(nkeys, 0);
    seg_runs.assign(nkeys, 0);
    SB_TRY(out.alloc(nnz));
    if (nnz == 0 || nc == 0) return SB_OK;
    if (nkeys > 0x7FFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "gather: block x panel key exceeds 31 bits");
    DevBuf<u32> keys, keys2;
    DevBuf<u64> payload, payload2, first, runs;
    SB_TRY(keys.alloc(nnz));
    SB_TRY(keys2.alloc(nnz));
    SB_TRY(payload.alloc(nnz));
    SB_TRY(payload2.alloc(nnz));
    SB_TRY(first.alloc(nkeys));
    SB_TRY(runs.alloc(nkeys));
    k_make_tkeys<<<ga_grid(nc * 32, 256, ctx), 256, 0, ctx->stream>>>(ptr_local, ent, nc, c0, mt->slot_of_gene.p, L.rows, L.npanels, keys.p, payload.p);
    count_launch(ctx);
    int end_bit = 1;
    while (end_bit < 32 && ((nkeys - 1) >> end_bit)) end_bit++;
    cub::DoubleBuffer<u32> dk(keys.p, keys2.p);
    cub::DoubleBuffer<u64> dv(payload.p, payload2.p);
    size_t tmp_bytes = 0;
    SB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, (unsigned long long)nnz, 0, end_bit, ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tmp_bytes));
    SB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, dk, dv, (unsigned long long)nnz, 0, end_bit, ctx->stream));
    count_launch(ctx, false);
    SB_CUDA(cudaMemsetAsync(first.p, 0xFF, nkeys * sizeof(u64), ctx->stream));
    SB_CUDA(cudaMemsetAsync(runs.p, 0, nkeys * sizeof(u64), ctx->stream));
    k_key_first<<<ga_grid(nnz, 256, ctx), 256, 0, ctx->stream>>>(dk.Current(), dv.Current(), nnz, first.p, (unsigned long long *)runs.p);
    k_unpack_u64<<<ga_grid(nnz, 256, ctx), 256, 0, ctx->stream>>>(dv.Current(), out.p, nnz);
    count_launch(ctx); count_launch(ctx);
    std::vector<u64> h(nkeys);
    SB_CUDA(cudaMemcpyAsync(h.data(), first.p, nkeys * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(seg_runs.data(), runs.p, nkeys * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    u64 next = nnz;
    for (u64 k = nkeys; k-- > 0;) {
        if (h[k] == ~0ull) h[k] = next;
        seg_len[k] = next - h[k];
        next = h[k];
    }
    return SB_OK;
}

// Units of the T side.  Every CTA owns one gene panel (or a few small ones) and sweeps the cell blocks in order, taking
// its share of each (block, panel) segment: the panel's rows of Y are staged once per CTA, no barrier separates units,
// and because all CTAs move through the cell blocks together the rows of T they reduce into stay in L2.
// CTAs are handed out to panels in proportion to their cost: entries plus GA_FLUSH_COST per run (a flush is ~25
// instructions and 20 reductions; the panels of rarely expressed genes have runs of one or two entries).
#define GA_FLUSH_COST 5.0
int gather_finish_t(sb_mat *mt, const std::vector<u64> &seg_len, const std::vector<u64> &seg_runs) {
    sb_ctx *ctx = mt->ctx;
    GatherLayout &L = mt->gt;
    u64 total_nnz = 0;
    for (u64 x : seg_len) total_nnz += x;
    L.nnz = total_nnz;
    std::vector<GUnit> units;
    std::vector<u32> first;
    mt->t_seg_len = seg_len;
    mt->t_seg_runs = seg_runs;
    mt->t_calibrated = 0;
    mt->t_rate.clear();
    const u32 per_cta = (u32)std::max(1, ctx->gather_items_per_cta);
    gather_units_t(seg_len, seg_runs, L.npanels, (u32)ctx->sm_count * per_cta, ctx->gather_flush_cost, units, first, ctx->gather_seg_cost);
    mt->t_units_host = units;
    mt->t_first_host = first;
    L.n_items = (u32)first.size() - 1;
    L.grid = std::min<u32>(L.n_items, (u32)ctx->sm_count);
    L.n_units = (u32)units.size();
    SB_TRY(L.units.alloc(units.size()));
    SB_TRY(L.cta_first.alloc(first.size()));
    if (!units.empty()) SB_CUDA(cudaMemcpyAsync(L.units.p, units.data(), units.size() * sizeof(GUnit), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(L.cta_first.p, first.data(), first.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    L.ent = L.ent_own.p;
    L.ready = true;
    return SB_OK;
}

// whole-shard T-side build from a cell-major pair (matrices created on the device; unpipelined uploads)
int gather_build_t(sb_mat *mt, const u64 *ptr, const uint2 *ent, u64 nnz) {
    if (mt->n > SB_GENE_MASK) {  // the packed entry keeps 22 bits for the cell: larger shards stay on the cell-major gather
        mt->gt.ready = false;
        return SB_OK;
    }
    SB_TRY(gather_assign_slots(mt, ent, nnz));
    std::vector<u64> seg, runs;
    SB_TRY(gather_build_t_range(mt, 0, mt->n, ptr, ent, nnz, mt->gt.ent_own, seg, runs));
    return gather_finish_t(mt, seg, runs);
}

// ---------------------------------------------------------------- T side: shares re-cut from a timed pass
// The static cost model (entries + flush_cost x runs) leaves the CTAs of one pass between 0.8x and 1.2x of the mean busy time
// (ncu: sm__cycles_active 1.19 / 1.49 / 1.79 M) and no setting of its constants does better (profiles/README.md).  What the model
// cannot know is how fast a given gene panel runs -- so the first product of a matrix is timed per CTA (clock64 around its work),
// every panel gets the measured cycles per unit of modelled cost of the CTAs that worked on it, and the cost line is cut again
// with those rates.  One D2H of `grid` counters and a host pass over the segment table, once per matrix.
int gather_recalibrate_t(sb_mat *mt, const long long *cycles_dev) {
    sb_ctx *ctx = mt->ctx;
    GatherLayout &L = mt->gt;
    mt->t_calibrated++;
    if (!L.ready || L.n_items != L.grid || mt->t_units_host.empty() || L.npanels == 0) return SB_OK;  // only the one-share-per-CTA form
    const u32 G = L.grid, np = L.npanels;
    std::vector<long long> cyc(2 * (size_t)G, 0);
    SB_CUDA(cudaMemcpyAsync(cyc.data(), cycles_dev, 2 * (size_t)G * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    const std::vector<u64> &seg_len = mt->t_seg_len, &seg_runs = mt->t_seg_runs;
    std::vector<u64> seg_pos(seg_len.size() + 1, 0);
    for (size_t k = 0; k < seg_len.size(); k++) seg_pos[k + 1] = seg_pos[k] + seg_len[k];
    // modelled cost of every CTA, split by panel
    std::vector<double> cta_cost(G, 0.0), pan_cost(np, 0.0), pan_time(np, 0.0);
    struct PanelShare { u32 panel; double cost, wgt; };
    std::vector<std::vector<PanelShare>> by_panel(G);
    for (u32 b = 0; b < G; b++) {
        for (u32 ui = mt->t_first_host[b]; ui < mt->t_first_host[b + 1]; ui++) {
            const GUnit &u = mt->t_units_host[ui];
            const size_t k = (size_t)(std::upper_bound(seg_pos.begin(), seg_pos.end(), u.begin) - seg_pos.begin()) - 1;
            if (k >= seg_len.size() || seg_len[k] == 0) continue;
            const double frac = (double)(u.end - u.begin) / (double)seg_len[k];
            const double c = frac * ((double)seg_len[k] + ctx->gather_flush_cost * (double)seg_runs[k] + ctx->gather_seg_cost);
            const double wgt = c * (mt->t_rate.size() == np ? mt->t_rate[u.panel] : 1.0);  // expected share of the CTA's time
            cta_cost[b] += wgt;
            if (by_panel[b].empty() || by_panel[b].back().panel != u.panel) by_panel[b].push_back({u.panel, 0.0, 0.0});
            by_panel[b].back().cost += c;
            by_panel[b].back().wgt += wgt;
        }
    }
    for (u32 b = 0; b < G; b++) {
        if (cta_cost[b] <= 0.0 || cyc[b] <= 0) continue;
        for (auto &pc : by_panel[b]) {  // a CTA's time is attributed to its panels in proportion to their expected share
            pan_cost[pc.panel] += pc.cost;
            pan_time[pc.panel] += (double)cyc[b] * pc.wgt / cta_cost[b];
        }
    }
    double tot_c = 0.0, tot_t = 0.0;
    for (u32 p = 0; p < np; p++) {
        tot_c += pan_cost[p];
        tot_t += pan_time[p];
    }
    if (const char *dump = getenv("SCANB200_GATHER_DUMP")) {  // diagnostics: per-CTA {index, SM, cycles, modelled cost, first panel}
        if (FILE *f = fopen(dump, "a")) {
            fprintf(f, "# round %d\n", mt->t_calibrated);
            for (u32 b = 0; b < G; b++)
                fprintf(f, "%u %lld %lld %.6g %u %zu\n", b, cyc[G + b], cyc[b], cta_cost[b], by_panel[b].empty() ? 0u : by_panel[b].front().panel, by_panel[b].size());
            fclose(f);
        }
    }
    if (!(tot_c > 0.0) || !(tot_t > 0.0)) return SB_OK;
    const double mean_rate = tot_t / tot_c;
    std::vector<double> rate(np, 1.0);
    for (u32 p = 0; p < np; p++)
        if (pan_cost[p] > 0.0) rate[p] = std::min(4.0, std::max(0.25, (pan_time[p] / pan_cost[p]) / mean_rate));
    std::vector<GUnit> units;
    std::vector<u32> first;
    gather_units_t(seg_len, seg_runs, np, G, ctx->gather_flush_cost, units, first, ctx->gather_seg_cost, &rate);
    if ((u32)first.size() - 1 != G) return SB_OK;  // keep the old shares if the cut degenerated
    SB_TRY(L.units.alloc(units.size()));
    SB_TRY(L.cta_first.alloc(first.size()));
    if (!units.empty()) SB_CUDA(cudaMemcpyAsync(L.units.p, units.data(), units.size() * sizeof(GUnit), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(L.cta_first.p, first.data(), first.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));  // host temporaries
    L.n_units = (u32)units.size();
    mt->t_units_host.swap(units);
    mt->t_first_host.swap(first);
    mt->t_rate = rate;
    if (TraceScope::on()) {
        double lo = 1e300, hi = 0.0;
        for (u32 b = 0; b < G; b++)
            if (cyc[b] > 0) { lo = std::min(lo, (double)cyc[b]); hi = std::max(hi, (double)cyc[b]); }
        fprintf(stderr, "[scanb200] gather T recalibrated: CTA cycles %.3g .. %.3g (mean rate %.3g per cost unit)\n", lo, hi, mean_rate);
    }
    return SB_OK;
}
