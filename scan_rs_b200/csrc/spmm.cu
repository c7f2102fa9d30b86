// spmm.cu -- the two sparse x dense-block products of the Krylov loop, with the normalization
// map fused into the load (the normalized matrix is never materialised) and the rank-1
// centring offset applied implicitly.
//
//   K7  spmm_t : T[c,:] = sum_g x_gc * Y[g,:] + v_c * (u^T Y)      cell-major gather
//       restates low_rank_offset.rs:83-96 -> mat.rs:1114-1133 -> prod.rs:56-81,154-214
//   K8  spmm_n : P[g,:] = sum_c x_gc * X[c,:] + u_g * (v^T X)      gene-major, cell-panelled gather
//       restates low_rank_offset.rs:68-81 -> mat.rs:1074-1090 -> prod.rs:30-51,87-148
//
// Lane mapping (both kernels): a dense row of the w-wide block is covered by LPR lanes holding
// two f64 columns each (one 16-byte load), so a warp works on G = 32/LPR nonzeros per step
// (w = 20 -> LPR = 10, G = 3, 30 of 32 lanes busy).  The per-nonzero scalars (map value, index)
// are computed once per nonzero by the lane that loaded it and handed to the column lanes through
// a 512-byte per-warp staging buffer in shared memory.
#include <type_traits>

#include "common.cuh"
#include "map.cuh"

#define FULLMASK 0xffffffffu

struct __align__(16) StageEnt {
    double x;
    u32 idx;
    u32 pad;
};

// ---------------------------------------------------------------- column sums:  out[j] = sum_r wgt[r] * A[r, j]
#define CS_ROWS_PER_BLOCK 512
#define CS_FINAL_THREADS 256
__global__ void k_colsum_partial(const double *__restrict__ A, u64 rows, u32 w, u32 ld, const double *__restrict__ wgt,
                                 double *__restrict__ partial) {
    // block b sums rows [b*CS, (b+1)*CS); thread t handles column t % w for rows t / w + k * (blockDim / w)
    extern __shared__ double sh[];
    u32 tpr = w;  // threads per row
    u32 rows_par = blockDim.x / tpr;
    u32 col = threadIdx.x % tpr, rsub = threadIdx.x / tpr;
    u64 r0 = (u64)blockIdx.x * CS_ROWS_PER_BLOCK;
    u64 r1 = min(rows, r0 + CS_ROWS_PER_BLOCK);
    double acc = 0.0;
    if (rsub < rows_par)
        for (u64 r = r0 + rsub; r < r1; r += rows_par) {
            double a = A[r * ld + col];
            acc += wgt ? wgt[r] * a : a;
        }
    sh[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x < tpr) {
        double s = 0.0;
        for (u32 k = 0; k < rows_par; k++) s += sh[k * tpr + threadIdx.x];
        partial[(u64)blockIdx.x * w + threadIdx.x] = s;
    }
}

// one block per column: strided sums of the partials, then a fixed-order tree (deterministic)
__global__ void __launch_bounds__(CS_FINAL_THREADS) k_colsum_final(const double *__restrict__ partial, u32 nblocks, u32 w, double *__restrict__ out) {
    __shared__ double sh[CS_FINAL_THREADS];
    const u32 j = blockIdx.x;
    double s = 0.0;
    for (u32 b = threadIdx.x; b < nblocks; b += CS_FINAL_THREADS) s += partial[(u64)b * w + j];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (u32 o = CS_FINAL_THREADS / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[j] = sh[0];
}

// deterministic two-stage weighted column sum; out is a device vector of w doubles
int colsum_weighted(sb_ctx *ctx, const double *A, u64 rows, u32 w, u32 ld, const double *wgt, double *out) {
    if (w == 0) return SB_OK;
    if (rows == 0) {
        SB_CUDA(cudaMemsetAsync(out, 0, w * sizeof(double), ctx->stream));
        return SB_OK;
    }
    u32 nblocks = cdiv(rows, CS_ROWS_PER_BLOCK);
    void *scr;
    SB_TRY(ctx_scratch(ctx, (size_t)nblocks * w * sizeof(double), &scr));
    if (w > 1024) return sb_fail(SB_ERR_UNSUPPORTED, "block width %u > 1024", w);
    int rows_par = 256 / (int)w;
    if (rows_par < 1) rows_par = 1;
    int threads = rows_par * (int)w;
    k_colsum_partial<<<nblocks, threads, threads * sizeof(double), ctx->stream>>>(A, rows, w, ld, wgt, (double *)scr);
    k_colsum_final<<<w, CS_FINAL_THREADS, 0, ctx->stream>>>((double *)scr, nblocks, w, out);
    count_launch(ctx); count_launch(ctx);
    return SB_OK;
}

// ---------------------------------------------------------------- K7: cell-major gather
// One warp per cell.  Kind-1 maps use a per-cell table of the 32 most common map values
// (lane l holds log_b(cs * (l+1) + 1)); it is the same function of the same inputs as the direct
// evaluation, so the bits are identical.
template <int LPR_T>
__global__ void __launch_bounds__(256) k_spmm_t(const u64 *__restrict__ cm_ptr, const uint2 *__restrict__ cm, u64 n, MapDev mp,
                                                const double *__restrict__ Y, u32 ldy, u32 col0, u32 wt, u32 w,
                                                const double *__restrict__ uy, const double *__restrict__ v,
                                                double *__restrict__ out, u32 ldo, int lpr_rt) {
    __shared__ StageEnt stage_all[8][32];
    const int LPR = LPR_T > 0 ? LPR_T : lpr_rt;
    const int G = 32 / LPR;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int grp = lane / LPR, lig = lane - grp * LPR;
    const bool lane_on = grp < G;
    StageEnt *stage = stage_all[wib];
    const u32 c_lo = col0 + 2 * lig;  // first of this lane's two columns
    const u64 warp = (u64)blockIdx.x * (blockDim.x >> 5) + wib;
    const u64 nwarps = (u64)gridDim.x * (blockDim.x >> 5);
    const bool pow2 = (LPR & (LPR - 1)) == 0;

    for (u64 c = warp; c < n; c += nwarps) {
        const u64 s = cm_ptr[c], e = cm_ptr[c + 1];
        const double cp = mp.col[c];
        double lut = 0.0;
        if (mp.kind == 1) lut = map_log_part(mp.log_base, cp, (u32)lane + 1u, sb_log_table);
        double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0;
        for (u64 k0 = s; k0 < e; k0 += 32) {
            const u64 k = k0 + lane;
            const bool valid = k < e;
            uint2 z = valid ? cm[k] : make_uint2(0u, 1u);
            double x;
            if (mp.kind == 1) {
                x = __shfl_sync(FULLMASK, lut, (int)((z.y - 1u) & 31u));
                if (z.y - 1u >= 32u) x = map_log_part(mp.log_base, cp, z.y, sb_log_table);
                if (mp.row) x = mp.row[z.x] * x;
            } else {
                x = map_full(mp, z.y, z.x, cp, true, sb_log_table);
            }
            __syncwarp();
            stage[lane].x = valid ? x : 0.0;
            stage[lane].idx = z.x;
            __syncwarp();
            const int cnt = (int)min((u64)32, e - k0);
            if (lane_on) {
                int t = grp;
                for (; t + G < cnt; t += 2 * G) {
                    const StageEnt m0 = stage[t], m1 = stage[t + G];
                    const double2 y0 = __ldg(reinterpret_cast<const double2 *>(Y + (size_t)m0.idx * ldy + c_lo));
                    const double2 y1 = __ldg(reinterpret_cast<const double2 *>(Y + (size_t)m1.idx * ldy + c_lo));
                    a0 = fma(m0.x, y0.x, a0);
                    a1 = fma(m0.x, y0.y, a1);
                    b0 = fma(m1.x, y1.x, b0);
                    b1 = fma(m1.x, y1.y, b1);
                }
                if (t < cnt) {
                    const StageEnt m0 = stage[t];
                    const double2 y0 = __ldg(reinterpret_cast<const double2 *>(Y + (size_t)m0.idx * ldy + c_lo));
                    a0 = fma(m0.x, y0.x, a0);
                    a1 = fma(m0.x, y0.y, a1);
                }
            }
        }
        a0 += b0;
        a1 += b1;
        // combine the G groups into group 0
        if (pow2) {
            for (int off = 16; off >= LPR; off >>= 1) {
                a0 += __shfl_xor_sync(FULLMASK, a0, off);
                a1 += __shfl_xor_sync(FULLMASK, a1, off);
            }
        } else {
            double t0 = a0, t1 = a1;
            for (int g = 1; g < G; g++) {
                double o0 = __shfl_down_sync(FULLMASK, a0, g * LPR);
                double o1 = __shfl_down_sync(FULLMASK, a1, g * LPR);
                t0 += o0;
                t1 += o1;
            }
            a0 = t0;
            a1 = t1;
        }
        if (grp == 0 && c_lo < col0 + wt) {
            double vc = v ? v[c] : 1.0;
            double o0 = a0, o1 = a1;
            if (uy) {
                o0 += vc * uy[c_lo];
                if (c_lo + 1 < w) o1 += vc * uy[c_lo + 1];
            }
            double *dst = out + (size_t)c * ldo + c_lo;
            const bool two = c_lo + 1 < col0 + wt && c_lo + 1 < w;
            if (two) {
                *reinterpret_cast<double2 *>(dst) = make_double2(o0, o1);
            } else {
                dst[0] = o0;
            }
        }
    }
}

// ---------------------------------------------------------------- K8: gene-major panel gather
// A CTA owns a contiguous run of work units; a unit is an nnz sub-range of one cell panel.  The
// panel's rows of X (pc x wt doubles) and its per-cell map parameters are staged in shared
// memory once per panel.  Each warp walks a contiguous span of the unit's entries, 32 at a time:
// the lane that loaded an entry evaluates its map value once and publishes {value, smem offset of
// the X row, gene} in the warp's staging buffer; then G = 32/LPR lane groups consume G entries per
// step (one 16-byte LDS of the X row + two DFMA per lane).  Entries are sorted by gene; a ballot
// of "gene differs from the previous entry" gives a warp-uniform head mask, so steps without a
// head are branch-free and a head flushes every group's partial row into P with f64 reductions
// (RED.ADD.F64) -- a few per (gene, panel), never one per nonzero.
struct __align__(16) StageN {
    double x;
    u32 off;   // byte offset of the X row inside the staged panel
    u32 gene;
};

template <int LPR_T>
__global__ void __launch_bounds__(1024, 1)  // <= 64 registers
k_spmm_n(const uint2 *__restrict__ gm, const u64 *__restrict__ gm_base, u32 np, u32 ur, u32 pc, u64 n, MapDev mp,
         const double *__restrict__ X, u32 ldx, u32 col0, u32 wt, u32 w, double *__restrict__ P, u32 ldp, int lpr_rt) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int LPR = LPR_T > 0 ? LPR_T : lpr_rt;
    const int G = 32 / LPR;
    const u32 wtp = 2 * LPR;
    double *Xs = reinterpret_cast<double *>(smem_raw);                   // pc * wtp
    double *cs = Xs + (size_t)pc * wtp;                                   // pc
    LogEnt *ltab = reinterpret_cast<LogEnt *>(cs + pc);                   // 128
    StageN *stage_all = reinterpret_cast<StageN *>(ltab + 128);          // nwarps * 32
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int grp = lane / LPR, lig = lane - grp * LPR;
    const bool lane_on = grp < G;
    StageN *stage = stage_all + wib * 32;
    const u32 xs_sa = (u32)__cvta_generic_to_shared(Xs) + (u32)lig * 16u;          // this lane's column pair in row 0
    const u32 stage_sa = (u32)__cvta_generic_to_shared(stage);
    const u32 stage_sa_own = stage_sa + (u32)lane * 16u;
    const u32 grp_bytes = (u32)grp * 16u;
    const u32 grp_bytes_safe = (u32)(lane_on ? grp : 0) * 16u;  // spare lanes shadow group 0
    const u32 c_lo = col0 + 2 * lig;
    const bool col_ok0 = lane_on && c_lo < col0 + wt && c_lo < w;
    const bool col_ok1 = lane_on && c_lo + 1 < col0 + wt && c_lo + 1 < w;
    const u32 NONE = 0xFFFFFFFFu;

    for (int i = threadIdx.x; i < 128; i += blockDim.x) ltab[i] = sb_log_table[i];

    const u64 total_units = (u64)np * ur;
    const u64 upc = (total_units + gridDim.x - 1) / gridDim.x;
    const u64 u_lo = (u64)blockIdx.x * upc;
    const u64 u_hi = min(total_units, u_lo + upc);
    u32 staged = NONE;

    for (u64 unit = u_lo; unit < u_hi; unit++) {
        const u32 p = (u32)(unit / ur), r = (u32)(unit % ur);
        if (p != staged) {
            __syncthreads();
            const u64 cell0 = (u64)p * pc;
            const u32 pcn = (u32)min((u64)pc, n - cell0);
            const u32 halfw = wtp / 2;
            for (u32 i = threadIdx.x; i < pcn * halfw; i += blockDim.x) {
                const u32 cl = i / halfw, j2 = (i - cl * halfw) * 2;
                const u32 col = col0 + j2;
                double2 val = make_double2(0.0, 0.0);
                // ldx is even and col is even, so col < w <= ldx implies col + 1 < ldx
                if (col < w) val = *reinterpret_cast<const double2 *>(X + (cell0 + cl) * (size_t)ldx + col);
                *reinterpret_cast<double2 *>(Xs + (size_t)cl * wtp + j2) = val;
            }
            for (u32 i = threadIdx.x; i < pcn; i += blockDim.x) cs[i] = mp.col[cell0 + i];
            staged = p;
            __syncthreads();
        }
        const u64 pb = gm_base[p], pe = gm_base[p + 1], plen = pe - pb;
        const u64 ub = pb + plen * r / ur, ue = pb + plen * (r + 1) / ur;
        // contiguous span per warp, multiple of 32 entries
        u64 span = (ue - ub + nw - 1) / nw;
        span = (span + 31) & ~(u64)31;
        const u64 wb = min(ue, ub + (u64)wib * span), we = min(ue, wb + span);

        u32 cur_gene = NONE, carry = NONE;  // warp-uniform
        double a0 = 0.0, a1 = 0.0;

        auto flush = [&]() {
            if (cur_gene != NONE) {
                if (col_ok0 && a0 != 0.0) atomicAdd(P + (size_t)cur_gene * ldp + c_lo, a0);
                if (col_ok1 && a1 != 0.0) atomicAdd(P + (size_t)cur_gene * ldp + c_lo + 1, a1);
            }
            a0 = 0.0;
            a1 = 0.0;
        };
        // entry t of the staging buffer: one 16-byte LDS for {x, off, gene}, one for the X row
        auto accumulate = [&](u32 t_bytes) {
            u32 m0, m1, off, g;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(m0), "=r"(m1), "=r"(off), "=r"(g) : "r"(stage_sa + t_bytes));
            double x0, x1;
            asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x0), "=d"(x1) : "r"(xs_sa + off));
            const double xm = __hiloint2double((int)m1, (int)m0);
            a0 = fma(xm, x0, a0);
            a1 = fma(xm, x1, a1);
        };

        for (u64 k0 = wb; k0 < we; k0 += 32) {
            const u64 k = k0 + lane;
            const bool valid = k < we;
            const uint2 z = valid ? __ldcs(gm + k) : make_uint2(NONE, 0u);
            const u32 gene = z.x & SB_GENE_MASK, cl = z.x >> SB_GENE_BITS;
            double x = 0.0;
            if (valid) x = map_full(mp, z.y, gene, cs[cl], false, ltab);
            u32 prev = __shfl_up_sync(FULLMASK, gene, 1);
            if (lane == 0) prev = carry;
            const u32 H = __ballot_sync(FULLMASK, valid && gene != prev);
            const int cnt = (we - k0) >= 32 ? 32 : (int)(we - k0);
            carry = __shfl_sync(FULLMASK, gene, cnt - 1);
            __syncwarp();
            asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(stage_sa_own), "r"((u32)__double2loint(x)), "r"((u32)__double2hiint(x)),
                         "r"(cl * wtp * 8u), "r"(gene)
                         : "memory");
            __syncwarp();
            if (LPR_T > 0 && cnt == 32 && H == 0u) {
                // whole chunk inside one gene segment: branch-free.  Lanes of the spare group (lane >= G*LPR) run
                // along on in-bounds addresses; their accumulators are never flushed.
                constexpr int GG = LPR_T > 0 ? 32 / LPR_T : 1;
#pragma unroll
                for (int st = 0; st < 32 / GG; st++) accumulate((u32)(st * GG) * 16u + grp_bytes_safe);
                if ((32 % GG) != 0 && grp < (32 % GG)) accumulate((u32)((32 / GG) * GG) * 16u + grp_bytes);
            } else {
                const u32 gmask = (1u << G) - 1u;
                for (int t0 = 0; t0 < cnt; t0 += G) {
                    const u32 hb = (H >> t0) & gmask;
                    if (hb == 0u) {
                        if (lane_on && t0 + grp < cnt) accumulate((u32)t0 * 16u + grp_bytes);
                    } else {
                        for (int j = 0; j < G; j++) {
                            if ((hb >> j) & 1u) {
                                flush();
                                cur_gene = stage[t0 + j].gene;
                            }
                            if (lane_on && grp == j && t0 + j < cnt) accumulate((u32)(t0 + j) * 16u);
                        }
                    }
                }
            }
        }
        flush();
    }
}

// P[g,j] = row_scale[g] * P[g,j] + u[g] * vx[j]   (kind-1 row scale is factored out of the sum)
__global__ void k_spmm_n_finalize(double *__restrict__ P, u32 m, u32 w, u32 ldp, const double *__restrict__ row,
                                  const double *__restrict__ u, const double *__restrict__ vx) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 total = (u64)m * w;
    if (i < total) {
        u32 g = (u32)(i / w), j = (u32)(i % w);
        double p = P[(size_t)g * ldp + j];
        if (row) p = row[g] * p;
        if (u) p += u[g] * vx[j];
        P[(size_t)g * ldp + j] = p;
    }
}

static MapDev make_map(const sb_nmat *a) {
    MapDev mp;
    mp.kind = a->kind;
    mp.log_base = a->log_base;
    mp.col = a->col_scale.p;
    mp.row = (a->kind == 1) ? (a->has_row_scale ? a->row_scale.p : nullptr) : a->row_scale.p;
    mp.l1 = a->kind == 1 ? a->l1c.p : nullptr;
    mp.inv_l1 = a->kind == 1 ? a->inv_l1c.p : nullptr;
    return mp;
}

template <typename F>
static void dispatch_lpr(int lpr, F &&f) {
    switch (lpr) {
    case 10: f(std::integral_constant<int, 10>()); break;
    case 16: f(std::integral_constant<int, 16>()); break;
    case 25: f(std::integral_constant<int, 25>()); break;
    case 32: f(std::integral_constant<int, 32>()); break;
    default: f(std::integral_constant<int, 0>()); break;
    }
}

// bytes / flops of one pass of width w over this shard (SURVEY.md 8d)
static void account(sb_ctx *ctx, const sb_mat *mt, u32 w, bool is_t) {
    double bytes = 8.0 * mt->nnz + 8.0 * (mt->n + 1) + 8.0 * w * ((double)mt->n + mt->m) + 8.0 * ((double)mt->m + mt->n);
    double flops = 2.0 * w * (double)mt->nnz;
    if (is_t) {
        ctx->prof.spmm_t_bytes += bytes;
        ctx->prof.spmm_t_flops += flops;
        ctx->prof.spmm_t_launches++;
    } else {
        ctx->prof.spmm_n_bytes += bytes;
        ctx->prof.spmm_n_flops += flops;
        ctx->prof.spmm_n_launches++;
    }
}

int mat_ensure_full_gm(sb_mat *mt);
// planes.cu
int planes_t(sb_nmat *a, const double *Y, u32 ldy, u32 w, double *out, u32 ldo, const GatherLayout *gl, const MapDev *mp, long long *cycles);
int planes_n(sb_nmat *a, const double *X, u32 ldx, u32 w, double *P, u32 ldp);
// gather.cu
int gather_run(sb_ctx *ctx, const GatherLayout &L, int mode, const MapDev &mp, u64 n_cells, const double *B, u32 ldb, u32 w, double *out, u32 ldo,
               long long *cycles = nullptr);
int gather_recalibrate_t(sb_mat *mt, const long long *cycles_dev);
int gather_t_init(sb_ctx *ctx, double *out, u64 n, u32 w, u32 ldo, const double *uy, const double *v);
// the panelled gather layouts cover the cold entries of a hybrid matrix, or every entry of a matrix without planes
static bool gather_usable(const sb_nmat *a, const GatherLayout &L) {
    const sb_mat *mt = a->mat;
    return mt->ctx->use_gather && L.ready && ((a->kind == 1 && mt->gd > 0) || mt->gd == 0);
}

// K7 driver: out[n x w] (ld ldo) = A^T . Y[m x w] (ld ldy) + v (u^T Y).  uy_scratch: device vector of >= w doubles.
int spmm_t(sb_nmat *a, const double *Y, u32 ldy, u32 w, double *out, u32 ldo, double *uy_scratch) {
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    if ((ldy & 1) || (ldo & 1)) return sb_fail(SB_ERR_INVALID_ARG, "spmm_t: leading dimensions must be even");
    const double *uy = nullptr;
    if (a->has_offset) {
        SB_TRY(colsum_weighted(ctx, Y, mt->m, w, ldy, a->u.p, uy_scratch));
        uy = uy_scratch;
    }
    if (mt->n == 0 || w == 0) return SB_OK;
    MapDev mp = make_map(a);
    ProfScope ps(ctx, PH_SPMM_T);
    // hybrid layout: the sparse kernel sees the cold entries only, the plane kernels add the rest
    const bool hybrid = a->kind == 1 && mt->gd > 0;
    if (gather_usable(a, mt->gt)) {
        // T = v (u^T Y)  ->  += planes (int8 tensor cores)  ->  += panelled gather of the sparse set (f64 reductions)
        SB_TRY(gather_t_init(ctx, out, mt->n, w, ldo, uy, a->v_ones ? nullptr : a->v.p));
        // first full-width product of this matrix: time every CTA of the gather, then re-cut its static shares (gather.cu)
        const bool calibrate = mt->t_calibrated < ctx->gather_calibrate && mt->gt.n_items == mt->gt.grid && w >= 8;
        DevBuf<long long> cyc;
        if (calibrate) {
            SB_TRY(cyc.alloc(2 * (size_t)mt->gt.grid));
            SB_CUDA(cudaMemsetAsync(cyc.p, 0, 2 * (size_t)mt->gt.grid * sizeof(long long), ctx->stream));
        }
        // plane kernels + log chain: the gather runs inside planes_t, per column pass, with its run factor L_c(1) deferred to the
        // reduction of the per-unit partial rows (planes.cu)
        const bool fused = hybrid && ctx->gather_defer && mp.kind == 1 && a->l1c.p;
        if (fused) {
            SB_TRY(planes_t(a, Y, ldy, w, out, ldo, &mt->gt, &mp, calibrate ? cyc.p : nullptr));
        } else {
            if (hybrid) SB_TRY(planes_t(a, Y, ldy, w, out, ldo, nullptr, nullptr, nullptr));
            SB_TRY(gather_run(ctx, mt->gt, 1, mp, mt->n, Y, ldy, w, out, ldo, calibrate ? cyc.p : nullptr));
        }
        if (calibrate) SB_TRY(gather_recalibrate_t(mt, cyc.p));
        account(ctx, mt, w, true);
        return SB_OK;
    }
    const u64 *cm_ptr = hybrid ? mt->cold_cm_ptr.p : mt->cm_ptr.p;
    const uint2 *cm = hybrid ? mt->cold_cm.p : mt->cm.p;
    const u32 tile_max = 64;
    u32 ntiles = (w + tile_max - 1) / tile_max;
    u32 tw = (w + ntiles - 1) / ntiles;
    tw = (tw + 1) & ~1u;
    int blocks = ctx->sm_count * 8;
    u64 need = (mt->n + 7) / 8;
    if ((u64)blocks > need) blocks = (int)need;
    for (u32 col0 = 0; col0 < w; col0 += tw) {
        u32 wt = min(tw, w - col0);
        int lpr = (int)((wt + 1) / 2);
        dispatch_lpr(lpr, [&](auto tag) {
            constexpr int L = decltype(tag)::value;
            k_spmm_t<L><<<blocks, 256, 0, ctx->stream>>>(cm_ptr, cm, mt->n, mp, Y, ldy, col0, wt, w, uy,
                                                         a->v_ones ? nullptr : a->v.p, out, ldo, lpr);
        });
        count_launch(ctx);
    }
    if (hybrid) SB_TRY(planes_t(a, Y, ldy, w, out, ldo, nullptr, nullptr, nullptr));
    account(ctx, mt, w, true);
    SB_CUDA(cudaGetLastError());
    return SB_OK;
}

// K8 driver: P[m x w] (ld ldp, with one extra row of ldp doubles at the end used for v^T X) =
// A . X[n x w] (ld ldx) + u (v^T X); all-reduced over ranks.
int spmm_n(sb_nmat *a, const double *X, u32 ldx, u32 w, double *P, u32 ldp) {
    sb_mat *mt = a->mat;
    sb_ctx *ctx = mt->ctx;
    if ((ldx & 1) || (ldp & 1)) return sb_fail(SB_ERR_INVALID_ARG, "spmm_n: leading dimensions must be even");
    double *vx = P + (size_t)mt->m * ldp;
    const u32 wpad = (w + 1) & ~1u;
    if (ctx->nranks > 1 && ldp != wpad) return sb_fail(SB_ERR_INVALID_ARG, "spmm_n: sharded runs need a contiguous output block");
    // zero the w (padded) columns of the m + 1 rows only: P may be a column block of a wider matrix
    SB_CUDA(cudaMemset2DAsync(P, (size_t)ldp * sizeof(double), 0, (size_t)wpad * sizeof(double), (size_t)mt->m + 1, ctx->stream));
    if (a->has_offset) SB_TRY(colsum_weighted(ctx, X, mt->n, w, ldx, a->v_ones ? nullptr : a->v.p, vx));
    MapDev mp = make_map(a);
    const bool hybrid = a->kind == 1 && mt->gd > 0;
    if (!hybrid) SB_TRY(mat_ensure_full_gm(mt));
    const uint2 *gm = hybrid ? mt->cold_gm.p : mt->gm.p;
    const u64 *gm_base = hybrid ? mt->cold_gm_base.p : mt->gm_base.p;
    const u64 sparse_nnz = hybrid ? mt->cold_nnz : mt->nnz;
    if (mt->nnz && w) {
        ProfScope ps(ctx, PH_SPMM_N);
        if (gather_usable(a, mt->gn)) {
            SB_TRY(gather_run(ctx, mt->gn, 0, mp, mt->n, X, ldx, w, P, ldp));
            if (hybrid) SB_TRY(planes_n(a, X, ldx, w, P, ldp));
            account(ctx, mt, w, false);
            SB_CUDA(cudaGetLastError());
        } else {
            // tile width: the X panel (pc x wt doubles) must fit in shared memory next to the staging buffers
            const size_t smem_budget = 200 * 1024;
            const int threads = 1024;
            size_t fixed = (size_t)mt->pc * 8 + 128 * sizeof(LogEnt) + (threads / 32) * 32 * sizeof(StageN);
            u32 tile_max = (u32)((smem_budget - fixed) / ((size_t)mt->pc * 8));
            tile_max &= ~1u;
            if (tile_max > 64) tile_max = 64;
            if (tile_max < 2) return sb_fail(SB_ERR_UNSUPPORTED, "spmm_n: panel does not fit in shared memory");
            u32 ntiles = (w + tile_max - 1) / tile_max;
            u32 tw = (w + ntiles - 1) / ntiles;
            tw = (tw + 1) & ~1u;
            u64 total_units = (u64)mt->np * mt->ur;
            for (u32 col0 = 0; col0 < w && sparse_nnz; col0 += tw) {
                u32 wt = min(tw, w - col0);
                int lpr = (int)((wt + 1) / 2);
                size_t smem = (size_t)mt->pc * (2 * lpr) * 8 + fixed;
                int ctas_per_sm = (int)std::min<size_t>(2, (220 * 1024) / smem);
                if (ctas_per_sm < 1) ctas_per_sm = 1;
                int blocks = ctx->sm_count * ctas_per_sm;
                if ((u64)blocks > total_units) blocks = (int)total_units;
                int rc = SB_OK;
                dispatch_lpr(lpr, [&](auto tag) {
                    constexpr int L = decltype(tag)::value;
                    cudaError_t e = cudaFuncSetAttribute(k_spmm_n<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                    if (e != cudaSuccess) {
                        rc = sb_fail(SB_ERR_CUDA, "cudaFuncSetAttribute(%zu B smem): %s", smem, cudaGetErrorString(e));
                        return;
                    }
                    k_spmm_n<L><<<blocks, threads, smem, ctx->stream>>>(gm, gm_base, mt->np, mt->ur, mt->pc, mt->n, mp, X, ldx, col0, wt, w, P, ldp, lpr);
                });
                SB_TRY(rc);
                count_launch(ctx);
            }
            if (hybrid) SB_TRY(planes_n(a, X, ldx, w, P, ldp));
            account(ctx, mt, w, false);
            SB_CUDA(cudaGetLastError());
        }
    }
    SB_TRY(comm_allreduce_f64(ctx, P, ((size_t)mt->m + 1) * ldp));
    const bool need_row = mp.kind == 1 && mp.row != nullptr;
    if (mt->m && w && (need_row || a->has_offset)) {
        k_spmm_n_finalize<<<cdiv((u64)mt->m * w, 256), 256, 0, ctx->stream>>>(P, mt->m, w, ldp, mp.kind == 1 ? mp.row : nullptr,
                                                                              a->has_offset ? a->u.p : nullptr, vx);
        count_launch(ctx);
    }
    return SB_OK;
}
