// matrix.cu -- device-resident count matrix: upload, the two device layouts, integer
// reductions (K1-K4, K6 of SURVEY.md 2.1), selection and download.
//
// Layouts (DESIGN.md "Data layout in HBM"):
//   cell-major  cm_ptr[n+1] (u64), cm[nnz] = {gene, count}                      8 B / nnz
//   gene-major, cell-panelled: panels of `pc` cells; inside a panel entries sorted by
//   (gene, cell); gm[k] = {gene | cell_local << 22, count}                      8 B / nnz
#include <cub/cub.cuh>

#include <algorithm>
#include <cmath>
#include <memory>
#include <numeric>

#include "common.cuh"

// gather.cu
int gather_build_n(sb_mat *mt, GatherLayout &L, const uint2 *gm, const u64 *gm_base_dev, u64 nnz);
int gather_build_t(sb_mat *mt, const u64 *ptr, const uint2 *ent, u64 nnz);
int gather_assign_slots(sb_mat *mt, const uint2 *ent, u64 nnz);
int gather_build_t_range(sb_mat *mt, u64 c0, u64 nc, const u64 *ptr_local, const uint2 *ent, u64 nnz, DevBuf<uint2> &out, std::vector<u64> &seg_len,
                         std::vector<u64> &seg_runs);
int gather_finish_t(sb_mat *mt, const std::vector<u64> &seg_len, const std::vector<u64> &seg_runs);
// planes.cu
int planes_select(sb_mat *mt, u64 c0, u64 c1);
int planes_split_launch(sb_mat *mt, u64 c0, u64 nc, const u64 *new_ptr, u32 *counts, uint2 *out);

// ---------------------------------------------------------------- small kernels
__global__ void k_interleave(const u32 *__restrict__ idx, const u32 *__restrict__ cnt, uint2 *__restrict__ out, u64 nnz) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 stride = (u64)gridDim.x * blockDim.x;
    for (; i < nnz; i += stride) out[i] = make_uint2(idx[i], cnt[i]);
}

// compact host form (sb_upload_compact): u16 gene index + u8 count; tracks the largest index for validation
__global__ void k_expand16(const unsigned short *__restrict__ idx, const unsigned char *__restrict__ cnt, uint2 *__restrict__ out, u64 nnz,
                           u32 *max_out) {
    u32 mx = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (u64)gridDim.x * blockDim.x) {
        const u32 g = idx[i];
        out[i] = make_uint2(g, (u32)cnt[i]);
        mx = max(mx, g);
    }
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(max_out, mx);
}

// packed host form (sb_upload_packed): one byte of gene delta + one nibble of count per entry.  One warp per cell rebuilds the
// gene indices with a segmented prefix sum: a delta of 0 marks an escape, whose absolute gene index is looked up in the sorted
// side list (esc_pos, esc_gene) and restarts the sum.  The first entry of a cell is a delta from -1.  Count nibbles of 15 are
// patched afterwards from the big-count side list (k_patch_big).  bad: 1 = escape without a side-list record, 2 = an escape's
// gene does not ascend.
__global__ void k_expand_packed(const u64 *__restrict__ ptr, u64 c0, u64 c1, const unsigned char *__restrict__ dgene,
                                const unsigned char *__restrict__ cnt4, const u64 *__restrict__ esc_pos, const u32 *__restrict__ esc_gene,
                                u64 n_esc, uint2 *__restrict__ out, u32 *max_out, int *bad) {
    const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    const u32 lane = threadIdx.x & 31;
    u32 mx = 0;
    for (u64 c = c0 + warp; c < c1; c += nwarps) {
        const u64 s = ptr[c], e = ptr[c + 1];
        u32 carry = 0xFFFFFFFFu;  // gene of the previous entry (-1 before the first)
        for (u64 base = s; base < e; base += 32) {
            const u64 k = base + lane;
            const bool valid = k < e;
            u32 v = valid ? (u32)dgene[k] : 0u;
            int f = valid && v == 0u;
            if (f) {
                u64 lo = 0, hi = n_esc;
                while (lo < hi) {
                    const u64 mid = (lo + hi) >> 1;
                    if (esc_pos[mid] < k) lo = mid + 1;
                    else hi = mid;
                }
                if (lo < n_esc && esc_pos[lo] == k) v = esc_gene[lo];
                else *bad = 1;
            }
            const bool esc = f;
#pragma unroll
            for (u32 o = 1; o < 32; o <<= 1) {
                const u32 vu = __shfl_up_sync(0xffffffffu, v, o);
                const int fu = __shfl_up_sync(0xffffffffu, f, o);
                if (lane >= o && !f) {
                    v += vu;
                    f = fu;
                }
            }
            if (!f) v += carry;
            u32 prev = __shfl_up_sync(0xffffffffu, v, 1);
            if (lane == 0) prev = carry;
            if (esc && k > s && v <= prev) *bad = 2;
            if (valid) {
                const u32 byte = cnt4[k >> 1];
                out[k] = make_uint2(v, (k & 1) ? byte >> 4 : byte & 15u);
                mx = max(mx, v);
            }
            carry = __shfl_sync(0xffffffffu, v, 31);
        }
    }
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0 && mx) atomicMax(max_out, mx);
}

// counts >= 255 of the compact form travel in a side list: entry big_pos[i] gets count big_cnt[i]
__global__ void k_patch_big(const u64 *__restrict__ big_pos, const u32 *__restrict__ big_cnt, u64 lo, u64 hi, uint2 *__restrict__ cm, u64 nnz) {
    u64 i = lo + (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < hi && big_pos[i] < nnz) cm[big_pos[i]].y = big_cnt[i];
}

// side-list positions of the packed form: ascending and below nnz (checked on the device -- the lists have millions of records)
__global__ void k_check_positions(const u64 *__restrict__ pos, u64 n, u64 nnz, int *bad) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        if (pos[i] >= nnz || (i && pos[i] <= pos[i - 1])) *bad = 3;
}

__global__ void k_max_u32(const u32 *__restrict__ v, u64 n, u32 *out) {
    u32 mx = 0;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) mx = max(mx, v[i]);
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, mx);
}

// ptr must be non-decreasing with ptr[0] == 0; flags violations
__global__ void k_check_ptr(const u64 *__restrict__ ptr, u64 len, int *bad) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len && ptr[i] > ptr[i + 1]) *bad = 1;
    if (i == 0 && ptr[0] != 0) *bad = 1;
}

// one warp per major vector: expands the vector id of every entry and emits (key, payload)
//   mode 0: input cell-major (vec = cell): key = (cell / pc) * m + gene, payload = packed gene-major entry
//   mode 1: input gene-major (vec = gene): key = cell,                  payload = {gene, count}
__global__ void k_make_keys(const u64 *__restrict__ ptr, const uint2 *__restrict__ ent, u64 nvec, int mode, u32 m,
                            u32 pc, u32 *__restrict__ keys, u64 *__restrict__ payload) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 v = warp; v < nvec; v += nwarps) {
        u64 s = ptr[v], e = ptr[v + 1];
        for (u64 k = s + lane; k < e; k += 32) {
            uint2 z = ent[k];
            if (mode == 0) {
                u32 panel = (u32)(v / pc), cl = (u32)(v % pc);
                keys[k] = panel * m + z.x;
                payload[k] = ((u64)z.y << 32) | (u64)(z.x | (cl << SB_GENE_BITS));
            } else {
                keys[k] = z.x;  // cell
                payload[k] = ((u64)z.y << 32) | (u64)(u32)v;
            }
        }
    }
}

__global__ void k_unpack_payload(const u64 *__restrict__ payload, uint2 *__restrict__ out, u64 nnz) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (u64)gridDim.x * blockDim.x) {
        u64 p = payload[i];
        out[i] = make_uint2((u32)p, (u32)(p >> 32));
    }
}

__global__ void k_hist_u32(const u32 *__restrict__ keys, u64 nnz, u32 *__restrict__ hist) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (u64)gridDim.x * blockDim.x)
        atomicAdd(&hist[keys[i]], 1u);
}

__global__ void k_u32_to_u64(const u32 *__restrict__ in, u64 *__restrict__ out, u64 n) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) out[i] = in[i];
}

__global__ void k_panel_base(const u64 *__restrict__ cm_ptr, u64 n, u32 pc, u32 np, u64 *__restrict__ base) {
    u32 p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p <= np) {
        u64 c = (u64)p * pc;
        base[p] = cm_ptr[c < n ? c : n];
    }
}

// K1: per-cell totals, wrapping u32 (sqz/src/mat.rs:377-406 via normalization.rs:159,161)
__global__ void k_cell_totals(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, u32 *__restrict__ out) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        u64 s = ptr[c], e = ptr[c + 1];
        u32 acc = 0;
        for (u64 k = s + lane; k < e; k += 32) acc += cm[k].y;
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) out[c] = acc;
    }
}

// K2 / K6: per-gene u64 sums (mode 0: v, 1: v*v, 2: 1) with optional cell / gene masks (K4 sweeps).
// Integer adds commute, so the atomics are bit-exact.  Warp-level pre-aggregation is not
// needed for correctness; contention on the hottest genes is absorbed by the L2 atomic units.
__global__ void k_gene_sums(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, int mode,
                            const unsigned char *__restrict__ excl_cells, const unsigned char *__restrict__ excl_genes,
                            unsigned long long *__restrict__ out) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        if (excl_cells && excl_cells[c]) continue;
        u64 s = ptr[c], e = ptr[c + 1];
        for (u64 k = s + lane; k < e; k += 32) {
            uint2 z = cm[k];
            if (excl_genes && excl_genes[z.x]) continue;
            unsigned long long v = mode == 0 ? (unsigned long long)z.y : mode == 1 ? (unsigned long long)z.y * z.y : (z.y ? 1ull : 0ull);
            if (v) atomicAdd(&out[z.x], v);
        }
    }
}

// per-cell u64 sums over non-excluded genes (K4 column sweep)
__global__ void k_cell_sums_masked(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n,
                                   const unsigned char *__restrict__ excl_cells, const unsigned char *__restrict__ excl_genes,
                                   unsigned long long *__restrict__ out) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        unsigned long long acc = 0;
        if (!(excl_cells && excl_cells[c])) {
            u64 s = ptr[c], e = ptr[c + 1];
            for (u64 k = s + lane; k < e; k += 32) {
                uint2 z = cm[k];
                if (!(excl_genes && excl_genes[z.x])) acc += z.y;
            }
            for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        }
        if (lane == 0) out[c] = acc;
    }
}

// `s < threshold` on exact integer sums (sqz/src/mat.rs:784-799); sets *updated when a mask bit flips
__global__ void k_apply_threshold(const unsigned long long *__restrict__ sums, u64 n, double thr, unsigned char *__restrict__ excl,
                                  int *updated) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !excl[i] && (double)sums[i] < thr) {
        excl[i] = 1;
        *updated = 1;
    }
}

// select_rows pass: count / write entries whose gene survives the old->new map
__global__ void k_select_rows(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, const u32 *__restrict__ gene_map,
                              const u64 *__restrict__ new_ptr, u32 *__restrict__ counts, uint2 *__restrict__ out) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        u64 s = ptr[c], e = ptr[c + 1];
        u64 wpos = new_ptr ? new_ptr[c] : 0;
        u32 total = 0;
        for (u64 k0 = s; k0 < e; k0 += 32) {
            u64 k = k0 + lane;
            uint2 z = k < e ? cm[k] : make_uint2(0, 0);
            u32 ng = k < e ? gene_map[z.x] : 0xFFFFFFFFu;
            bool keep = ng != 0xFFFFFFFFu;
            unsigned mask = __ballot_sync(0xffffffffu, keep);
            if (out && keep) out[wpos + total + __popc(mask & ((1u << lane) - 1u))] = make_uint2(ng, z.y);
            total += __popc(mask);
        }
        if (counts && lane == 0) counts[c] = total;
    }
}

__global__ void k_gather_len(const u64 *__restrict__ ptr, const u64 *__restrict__ cols, u64 count, u32 *__restrict__ len) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) len[i] = (u32)(ptr[cols[i] + 1] - ptr[cols[i]]);
}

__global__ void k_select_cols(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, const u64 *__restrict__ cols, u64 count,
                              const u64 *__restrict__ new_ptr, uint2 *__restrict__ out) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 j = warp; j < count; j += nwarps) {
        u64 s = ptr[cols[j]], e = ptr[cols[j] + 1], d = new_ptr[j];
        for (u64 k = s + lane; k < e; k += 32) out[d + (k - s)] = cm[k];
    }
}

__global__ void k_split_entries(const uint2 *__restrict__ ent, u64 nnz, u32 *__restrict__ idx, u32 *__restrict__ cnt) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (u64)gridDim.x * blockDim.x) {
        uint2 z = ent[i];
        idx[i] = z.x;
        cnt[i] = z.y;
    }
}

static inline int grid_for(u64 work_items, int threads, sb_ctx *ctx, int per_sm = 8) {
    u64 blocks = (work_items + threads - 1) / threads;
    u64 cap = (u64)ctx->sm_count * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

static inline int bits_for(u64 max_value) {
    int b = 1;
    while (b < 64 && (max_value >> b)) b++;
    return b;
}

// stable radix sort of (u32 key, u64 payload); result in keys / payload (buffers may be swapped)
static int sort_pairs(sb_ctx *ctx, DevBuf<u32> &keys, DevBuf<u64> &payload, u64 count, int end_bit) {
    if (count == 0) return SB_OK;
    DevBuf<u32> keys2;
    DevBuf<u64> payload2;
    SB_TRY(keys2.alloc(count));
    SB_TRY(payload2.alloc(count));
    cub::DoubleBuffer<u32> dk(keys.p, keys2.p);
    cub::DoubleBuffer<u64> dv(payload.p, payload2.p);
    size_t tmp_bytes = 0;
    SB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dk, dv, (unsigned long long)count, 0, end_bit, ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tmp_bytes));
    SB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, dk, dv, (unsigned long long)count, 0, end_bit, ctx->stream));
    count_launch(ctx, false);
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (dk.Current() != keys.p) keys.swap(keys2);
    if (dv.Current() != payload.p) payload.swap(payload2);
    return SB_OK;
}

static int exclusive_scan_u32_to_u64(sb_ctx *ctx, const u32 *counts, u64 n, u64 *out_ptr /* n+1 */) {
    // out_ptr[0..n] = exclusive prefix sums, out_ptr[n] = total
    DevBuf<u64> wide;
    SB_TRY(wide.alloc(n + 1));
    SB_CUDA(cudaMemsetAsync(wide.p, 0, (n + 1) * sizeof(u64), ctx->stream));
    if (n) {
        k_u32_to_u64<<<grid_for(n, 256, ctx), 256, 0, ctx->stream>>>(counts, wide.p, n);
        count_launch(ctx);
    }
    size_t tmp_bytes = 0;
    SB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, wide.p, out_ptr, (unsigned long long)(n + 1), ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tmp_bytes));
    SB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, wide.p, out_ptr, (unsigned long long)(n + 1), ctx->stream));
    count_launch(ctx, false);
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// choose the panel geometry: panels of pc cells (power of two <= 1024) such that there are enough
// panels to spread over the SMs, and `ur` nnz-balanced work units per panel
static void choose_panels(sb_mat *mt) {
    sb_ctx *ctx = mt->ctx;
    u32 pc = SB_MAX_PANEL_CELLS;
    while (pc > 128 && (mt->n + pc - 1) / pc < (u64)ctx->sm_count) pc >>= 1;
    mt->pc = pc;
    mt->np = (u32)((mt->n + pc - 1) / pc);
    u64 target_units = (u64)ctx->sm_count * 8;
    u32 ur = mt->np ? (u32)((target_units + mt->np - 1) / mt->np) : 1;
    if (ur < 1) ur = 1;
    if (ur > 64) ur = 64;
    mt->ur = ur;
}

// ---- range-based building blocks (whole matrix or one upload chunk of whole cell panels) -------------------
// gene-major panelled order of `nc` cells given their (range-local) cell-major pair: stable sort by (panel, gene)
static int gene_major_range(sb_mat *mt, u64 nc, const u64 *ptr_local, const uint2 *ent, u64 nnz, DevBuf<uint2> &gm) {
    sb_ctx *ctx = mt->ctx;
    SB_TRY(gm.alloc(nnz));
    if (nnz == 0) return SB_OK;
    const u64 npanels = (nc + mt->pc - 1) / mt->pc;
    if (npanels * mt->m > 0xFFFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "panel x gene key exceeds 32 bits");
    DevBuf<u32> keys;
    DevBuf<u64> payload;
    SB_TRY(keys.alloc(nnz));
    SB_TRY(payload.alloc(nnz));
    k_make_keys<<<grid_for(nc * 32, 256, ctx, 16), 256, 0, ctx->stream>>>(ptr_local, ent, nc, 0, mt->m, mt->pc, keys.p, payload.p);
    count_launch(ctx);
    SB_TRY(sort_pairs(ctx, keys, payload, nnz, bits_for(npanels * mt->m - 1)));
    k_unpack_payload<<<grid_for(nnz, 256, ctx, 16), 256, 0, ctx->stream>>>(payload.p, gm.p, nnz);
    count_launch(ctx);
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

static int panel_base(sb_mat *mt, const u64 *cm_ptr, DevBuf<u64> &gm_base) {
    sb_ctx *ctx = mt->ctx;
    SB_TRY(gm_base.alloc((size_t)mt->np + 1));
    k_panel_base<<<cdiv(mt->np + 1, 256), 256, 0, ctx->stream>>>(cm_ptr, mt->n, mt->pc, mt->np, gm_base.p);
    count_launch(ctx);
    return SB_OK;
}

// the gene-major copy of ALL entries (binomial residual maps, which have no per-cell value table)
int mat_ensure_full_gm(sb_mat *mt) {
    if (mt->have_full_gm) return SB_OK;
    SB_TRY(panel_base(mt, mt->cm_ptr.p, mt->gm_base));
    SB_TRY(gene_major_range(mt, mt->n, mt->cm_ptr.p, mt->cm.p, mt->nnz, mt->gm));
    mt->have_full_gm = true;
    return SB_OK;
}

__global__ void k_add_offset(const u64 *__restrict__ src, u64 n, u64 add, u64 *__restrict__ dst) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i] + add;
}

// plane / cold split of local cells [c0, c1): sets their plane bits, returns the range-local cold pair
static int split_range(sb_mat *mt, u64 c0, u64 c1, DevBuf<u64> &ptr_local, DevBuf<uint2> &cold, u64 *cold_nnz) {
    sb_ctx *ctx = mt->ctx;
    const u64 nc = c1 - c0;
    DevBuf<u32> counts;
    SB_TRY(counts.alloc(nc));
    SB_TRY(ptr_local.alloc(nc + 1));
    SB_TRY(planes_split_launch(mt, c0, nc, nullptr, counts.p, nullptr));
    SB_TRY(exclusive_scan_u32_to_u64(ctx, counts.p, nc, ptr_local.p));
    SB_CUDA(cudaMemcpyAsync(cold_nnz, ptr_local.p + nc, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_TRY(cold.alloc(*cold_nnz));
    SB_TRY(planes_split_launch(mt, c0, nc, ptr_local.p, nullptr, cold.p));
    return SB_OK;
}

// whole-matrix hybrid build (matrices created on the device: generator, select, partition; gene-major uploads)
static int build_hybrid(sb_mat *mt) {
    sb_ctx *ctx = mt->ctx;
    SyncScope tr(ctx, "build: hybrid total");
    SB_TRY(planes_select(mt, 0, mt->n));
    if (mt->gd == 0) return SB_OK;
    {
        SyncScope t4(ctx, "build: split hot/cold");
        SB_TRY(split_range(mt, 0, mt->n, mt->cold_cm_ptr, mt->cold_cm, &mt->cold_nnz));
    }
    SyncScope t3(ctx, "build: cold gene-major sort");
    SB_TRY(panel_base(mt, mt->cold_cm_ptr.p, mt->cold_gm_base));
    SB_TRY(gene_major_range(mt, mt->n, mt->cold_cm_ptr.p, mt->cold_cm.p, mt->cold_nnz, mt->cold_gm));
    return SB_OK;
}

static int set_global_shape(sb_mat *mt) {
    sb_ctx *ctx = mt->ctx;
    std::vector<u64> all;
    SB_TRY(comm_allgather_u64_host(ctx, mt->n, all));
    mt->n_global = 0;
    mt->cell_offset = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        if (r < ctx->rank) mt->cell_offset += all[r];
        mt->n_global += all[r];
    }
    choose_panels(mt);
    return SB_OK;
}

// panelled gather layouts (gather.cu) over the sparse set the products use; whatever the upload pipeline has not built yet
static int finish_gather(sb_mat *mt) {
    SyncScope tr(mt->ctx, "build: gather layouts");
    const bool cold = mt->gd > 0;
    if (!mt->gn.ready)
        SB_TRY(gather_build_n(mt, mt->gn, cold ? mt->cold_gm.p : mt->gm.p, cold ? mt->cold_gm_base.p : mt->gm_base.p, cold ? mt->cold_nnz : mt->nnz));
    if (!mt->gt.ready)
        SB_TRY(gather_build_t(mt, cold ? mt->cold_cm_ptr.p : mt->cm_ptr.p, cold ? mt->cold_cm.p : mt->cm.p, cold ? mt->cold_nnz : mt->nnz));
    return SB_OK;
}

static int finish_matrix(sb_mat *mt) {
    SB_TRY(set_global_shape(mt));
    SB_TRY(build_hybrid(mt));
    if (mt->gd == 0) SB_TRY(mat_ensure_full_gm(mt));
    SB_TRY(finish_gather(mt));
    return SB_OK;
}

// The entries of an upload on the host, in the plain (u32 + u32) or the compact (u16 + u8 + side list) form, and their
// device staging buffers.
struct HostEntries {
    const u32 *idx32 = nullptr, *cnt32 = nullptr;
    const unsigned short *idx16 = nullptr;
    const unsigned char *cnt8 = nullptr;
    u64 n_big = 0;
    const u64 *big_pos = nullptr;
    const u32 *big_cnt = nullptr;
    bool compact = false;
    // packed form: gene deltas + count nibbles + two side lists (escaped genes; counts >= 15 share big_pos / big_cnt)
    bool packed = false;
    const unsigned char *dgene8 = nullptr, *cnt4 = nullptr;
    u64 n_esc = 0;
    const u64 *esc_pos = nullptr;
    const u32 *esc_gene = nullptr;
};
struct DevEntries {
    DevBuf<u32> idx32, cnt32, big_cnt, esc_gene;
    DevBuf<unsigned short> idx16;
    DevBuf<unsigned char> cnt8;  // packed form: the count nibbles
    DevBuf<unsigned char> dgene8;
    DevBuf<u64> big_pos, esc_pos;
    DevBuf<int> bad;             // packed form: decoder flags
    u64 nnz = 0;
    int alloc(const HostEntries &h, u64 nnz_, cudaStream_t st) {
        nnz = nnz_;
        if (h.packed) {
            SB_TRY(dgene8.alloc(nnz));
            SB_TRY(cnt8.alloc((nnz + 1) / 2));
            SB_TRY(big_pos.alloc(h.n_big));
            SB_TRY(big_cnt.alloc(h.n_big));
            SB_TRY(esc_pos.alloc(h.n_esc));
            SB_TRY(esc_gene.alloc(h.n_esc));
            SB_TRY(bad.alloc(1));
            SB_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), st));
            if (h.n_big) {
                SB_CUDA(cudaMemcpyAsync(big_pos.p, h.big_pos, h.n_big * sizeof(u64), cudaMemcpyHostToDevice, st));
                SB_CUDA(cudaMemcpyAsync(big_cnt.p, h.big_cnt, h.n_big * sizeof(u32), cudaMemcpyHostToDevice, st));
            }
            if (h.n_esc) {
                SB_CUDA(cudaMemcpyAsync(esc_pos.p, h.esc_pos, h.n_esc * sizeof(u64), cudaMemcpyHostToDevice, st));
                SB_CUDA(cudaMemcpyAsync(esc_gene.p, h.esc_gene, h.n_esc * sizeof(u32), cudaMemcpyHostToDevice, st));
                k_check_positions<<<(unsigned)std::min<u64>(cdiv(h.n_esc, 256), 2048), 256, 0, st>>>(esc_pos.p, h.n_esc, nnz, bad.p);
            }
            if (h.n_big) k_check_positions<<<(unsigned)std::min<u64>(cdiv(h.n_big, 256), 2048), 256, 0, st>>>(big_pos.p, h.n_big, nnz, bad.p);
        } else if (h.compact) {
            SB_TRY(idx16.alloc(nnz));
            SB_TRY(cnt8.alloc(nnz));
            SB_TRY(big_pos.alloc(h.n_big));
            SB_TRY(big_cnt.alloc(h.n_big));
            if (h.n_big) {
                SB_CUDA(cudaMemcpyAsync(big_pos.p, h.big_pos, h.n_big * sizeof(u64), cudaMemcpyHostToDevice, st));
                SB_CUDA(cudaMemcpyAsync(big_cnt.p, h.big_cnt, h.n_big * sizeof(u32), cudaMemcpyHostToDevice, st));
            }
        } else {
            SB_TRY(idx32.alloc(nnz));
            SB_TRY(cnt32.alloc(nnz));
        }
        return SB_OK;
    }
    void release() {
        idx32.release(); cnt32.release(); idx16.release(); cnt8.release(); big_pos.release(); big_cnt.release();
        dgene8.release(); esc_pos.release(); esc_gene.release(); bad.release();
    }
};

// host -> device copy of entries [e0, e1) on `st`
static int copy_entries(const HostEntries &h, DevEntries &d, u64 e0, u64 e1, cudaStream_t st) {
    if (e1 <= e0) return SB_OK;
    if (h.packed) {
        // two entries share a count byte: a chunk that starts on an odd entry re-copies the byte its predecessor ended in (same value)
        SB_CUDA(cudaMemcpyAsync(d.dgene8.p + e0, h.dgene8 + e0, e1 - e0, cudaMemcpyHostToDevice, st));
        SB_CUDA(cudaMemcpyAsync(d.cnt8.p + e0 / 2, h.cnt4 + e0 / 2, (e1 + 1) / 2 - e0 / 2, cudaMemcpyHostToDevice, st));
    } else if (h.compact) {
        SB_CUDA(cudaMemcpyAsync(d.idx16.p + e0, h.idx16 + e0, (e1 - e0) * sizeof(unsigned short), cudaMemcpyHostToDevice, st));
        SB_CUDA(cudaMemcpyAsync(d.cnt8.p + e0, h.cnt8 + e0, (e1 - e0), cudaMemcpyHostToDevice, st));
    } else {
        SB_CUDA(cudaMemcpyAsync(d.idx32.p + e0, h.idx32 + e0, (e1 - e0) * sizeof(u32), cudaMemcpyHostToDevice, st));
        SB_CUDA(cudaMemcpyAsync(d.cnt32.p + e0, h.cnt32 + e0, (e1 - e0) * sizeof(u32), cudaMemcpyHostToDevice, st));
    }
    return SB_OK;
}

// staged entries [e0, e1) -> interleaved {index, count} in `out` (same positions); largest index into *d_max
// (packed form: d_ptr is the device copy of the cell pointers and [c0, c1) the cells whose entries are [e0, e1))
static int expand_entries(sb_ctx *ctx, const HostEntries &h, DevEntries &d, u64 e0, u64 e1, uint2 *out, u32 *d_max, const u64 *d_ptr = nullptr,
                          u64 c0 = 0, u64 c1 = 0) {
    if (e1 <= e0) return SB_OK;
    const u64 cnt = e1 - e0;
    if (h.packed) {
        if (!d_ptr) return sb_fail(SB_ERR_INVALID_ARG, "expand_entries: the packed form needs the cell pointers");
        k_expand_packed<<<grid_for((c1 - c0) * 32, 256, ctx, 16), 256, 0, ctx->stream>>>(d_ptr, c0, c1, d.dgene8.p, d.cnt8.p, d.esc_pos.p, d.esc_gene.p,
                                                                                      h.n_esc, out, d_max, d.bad.p);
        count_launch(ctx);
        const u64 lo = std::lower_bound(h.big_pos, h.big_pos + h.n_big, e0) - h.big_pos;
        const u64 hi = std::lower_bound(h.big_pos, h.big_pos + h.n_big, e1) - h.big_pos;
        if (hi > lo) {
            k_patch_big<<<cdiv(hi - lo, 256), 256, 0, ctx->stream>>>(d.big_pos.p, d.big_cnt.p, lo, hi, out, d.nnz);
            count_launch(ctx);
        }
    } else if (h.compact) {
        k_expand16<<<grid_for(cnt, 256, ctx, 16), 256, 0, ctx->stream>>>(d.idx16.p + e0, d.cnt8.p + e0, out + e0, cnt, d_max);
        count_launch(ctx);
        const u64 lo = std::lower_bound(h.big_pos, h.big_pos + h.n_big, e0) - h.big_pos;
        const u64 hi = std::lower_bound(h.big_pos, h.big_pos + h.n_big, e1) - h.big_pos;
        if (hi > lo) {
            k_patch_big<<<cdiv(hi - lo, 256), 256, 0, ctx->stream>>>(d.big_pos.p, d.big_cnt.p, lo, hi, out, d.nnz);
            count_launch(ctx);
        }
    } else {
        k_max_u32<<<grid_for(cnt, 256, ctx), 256, 0, ctx->stream>>>(d.idx32.p + e0, cnt, d_max);
        k_interleave<<<grid_for(cnt, 256, ctx, 16), 256, 0, ctx->stream>>>(d.idx32.p + e0, d.cnt32.p + e0, out + e0, cnt);
        count_launch(ctx); count_launch(ctx);
    }
    return SB_OK;
}

// packed form: the decoder's flags (read after a synchronisation of the build stream)
static int packed_status(sb_ctx *ctx, const HostEntries &he, DevEntries &de) {
    if (!he.packed) return SB_OK;
    int h = 0;
    SB_CUDA(cudaMemcpyAsync(&h, de.bad.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (h == 1) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_packed: a zero gene delta has no record in the escape list");
    if (h == 3) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_packed: side-list positions must be ascending and below nnz");
    if (h) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_packed: an escaped gene index does not ascend inside its cell");
    return SB_OK;
}

// Cell-major upload as a pipeline: the host arrays are copied in chunks of whole cell panels on a second
// stream while the library stream turns the previous chunk into the device layouts (interleave, plane /
// cold split, per-chunk panel sort).  The planes are chosen from the first chunk (a sample of the cells).
static int upload_pipelined(sb_mat *mt, const u64 *h_indptr, const HostEntries &he, DevEntries &de, u32 *d_max) {
    sb_ctx *ctx = mt->ctx;
    const u64 n = mt->n;
    const u32 nch = (u32)std::max(1, ctx->upload_chunks);
    const u64 calign = std::max<u64>(mt->pc, GA_TBLOCK);  // whole cell panels and whole T-side cell blocks (pc divides GA_TBLOCK)
    u64 cells_per = ((n + nch - 1) / nch + calign - 1) / calign * calign;
    std::vector<u64> cb;
    for (u64 c = 0; c < n; c += cells_per) cb.push_back(c);
    cb.push_back(n);
    const size_t chunks = cb.size() - 1;
    if (!ctx->copy_stream) SB_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    std::vector<cudaEvent_t> ev(chunks);
    cudaEvent_t ready;
    SB_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    SB_CUDA(cudaEventRecord(ready, ctx->stream));  // the staging buffers exist (stream-ordered allocation)
    SB_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ready, 0));
    prof_begin(ctx, PH_UPLOAD);
    // The first chunk's build makes small host -> device copies of its own (hot-gene and slot tables); they queue on the
    // copy engine behind every bulk copy already issued, so only two chunks are in flight until that build is done.
    for (size_t i = 0; i < chunks; i++) SB_CUDA(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    size_t issued = 0;
    auto issue_copies = [&](size_t upto) -> int {
        for (; issued < std::min(upto, chunks); issued++) {
            const u64 e0 = h_indptr[cb[issued]], e1 = h_indptr[cb[issued + 1]];
            SB_TRY(copy_entries(he, de, e0, e1, ctx->copy_stream));
            SB_CUDA(cudaEventRecord(ev[issued], ctx->copy_stream));
        }
        return SB_OK;
    };
    SB_TRY(issue_copies(2));
    std::vector<DevBuf<u64>> ptrs(chunks);
    std::vector<DevBuf<uint2>> colds(chunks), gms(chunks), tps(chunks);
    std::vector<u64> cold_n(chunks, 0);
    std::vector<u64> seg_all, seg, runs_all, runs;
    const bool build_t = n <= SB_GENE_MASK;
    int rc = SB_OK;
    for (size_t i = 0; i < chunks && rc == SB_OK; i++) {
        const u64 c0 = cb[i], c1 = cb[i + 1], e0 = h_indptr[c0], e1 = h_indptr[c1];
        cudaStreamWaitEvent(ctx->stream, ev[i], 0);
        // Drain the build stream after every stage (the copies run on their own stream and are not held up).  Measured at
        // 1.3M cells: letting the host run ahead of the device makes the whole upload take ~390-510 ms instead of ~125 ms
        // (stream-ordered allocations issued long before the frees they could reuse have executed grow the pool).
        auto drain = [&]() { if (ctx->upload_sync) cudaStreamSynchronize(ctx->stream); };
        {
            SyncScope t0(ctx, "chunk: wait copy + expand");
            rc = expand_entries(ctx, he, de, e0, e1, mt->cm.p, d_max, mt->cm_ptr.p, c0, c1);
            drain();
            // indices are validated before any kernel uses them as table offsets
            u32 hmax = 0;
            if (rc == SB_OK && cudaMemcpyAsync(&hmax, d_max, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream) == cudaSuccess &&
                cudaStreamSynchronize(ctx->stream) == cudaSuccess && hmax >= mt->m)
                rc = sb_fail(SB_ERR_INVALID_ARG, "sb_upload: index %u out of range %u", hmax, mt->m);
            if (rc == SB_OK) rc = packed_status(ctx, he, de);
        }
        if (rc == SB_OK && i == 0) rc = planes_select(mt, c0, c1);
        if (rc == SB_OK && mt->gd > 0) {
            {
                SyncScope t1(ctx, "chunk: split hot/cold");
                rc = split_range(mt, c0, c1, ptrs[i], colds[i], &cold_n[i]);
                drain();
            }
            if (rc == SB_OK) {
                SyncScope t2(ctx, "chunk: cold gene-major sort");
                rc = gene_major_range(mt, c1 - c0, ptrs[i].p, colds[i].p, cold_n[i], gms[i]);
                drain();
            }
            if (rc == SB_OK && build_t) {
                SyncScope t3(ctx, "chunk: T-side order");
                if (i == 0) rc = gather_assign_slots(mt, colds[0].p, cold_n[0]);
                if (rc == SB_OK) rc = gather_build_t_range(mt, c0, c1 - c0, ptrs[i].p, colds[i].p, cold_n[i], tps[i], seg, runs);
                seg_all.insert(seg_all.end(), seg.begin(), seg.end());
                runs_all.insert(runs_all.end(), runs.begin(), runs.end());
                drain();
            }
        }
        if (rc == SB_OK) rc = issue_copies(chunks);  // after the first chunk: everything else
    }
    cudaStreamSynchronize(ctx->copy_stream);
    prof_end(ctx, PH_UPLOAD);  // spans the overlapped copies and builds
    for (auto e : ev) cudaEventDestroy(e);
    cudaEventDestroy(ready);
    SB_TRY(rc);
    if (mt->gd == 0) return SB_OK;
    SyncScope tcat(ctx, "upload: concatenate chunks");
    // concatenate the per-chunk cold layouts
    mt->cold_nnz = 0;
    for (u64 x : cold_n) mt->cold_nnz += x;
    SB_TRY(mt->cold_cm_ptr.alloc(n + 1));
    SB_TRY(mt->cold_cm.alloc(mt->cold_nnz));
    SB_TRY(mt->cold_gm.alloc(mt->cold_nnz));
    if (build_t) SB_TRY(mt->gt.ent_own.alloc(mt->cold_nnz));
    u64 base = 0;
    for (size_t i = 0; i < chunks; i++) {
        const u64 nc = cb[i + 1] - cb[i];
        k_add_offset<<<cdiv(nc + 1, 256), 256, 0, ctx->stream>>>(ptrs[i].p, nc + 1, base, mt->cold_cm_ptr.p + cb[i]);
        count_launch(ctx);
        if (cold_n[i]) {
            SB_CUDA(cudaMemcpyAsync(mt->cold_cm.p + base, colds[i].p, cold_n[i] * sizeof(uint2), cudaMemcpyDeviceToDevice, ctx->stream));
            SB_CUDA(cudaMemcpyAsync(mt->cold_gm.p + base, gms[i].p, cold_n[i] * sizeof(uint2), cudaMemcpyDeviceToDevice, ctx->stream));
            if (build_t)
                SB_CUDA(cudaMemcpyAsync(mt->gt.ent_own.p + base, tps[i].p, cold_n[i] * sizeof(uint2), cudaMemcpyDeviceToDevice, ctx->stream));
        }
        base += cold_n[i];
    }
    SB_TRY(panel_base(mt, mt->cold_cm_ptr.p, mt->cold_gm_base));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (build_t) SB_TRY(gather_finish_t(mt, seg_all, runs_all));
    return SB_OK;
}

// SCANB200_TRACE: state of the stream-ordered pool (reserved = held from the driver, used = handed out)
static void trace_pool(sb_ctx *ctx, const char *label) {
    if (!TraceScope::on()) return;
    cudaMemPool_t pool = ctx->pool;
    if (!pool) return;
    unsigned long long reserved = 0, used = 0;
    cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved);
    cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
    fprintf(stderr, "[scanb200] pool %-22s reserved %7.2f GB used %7.2f GB\n", label, reserved / 1e9, used / 1e9);
}

// Every rank of a sharded context must take the same turn before the collectives of an upload (global shape, hot-gene counts):
// a rank that rejected its own input would otherwise leave the others waiting inside them.
int agree_status(sb_ctx *ctx, int rc, const char *what) {
    if (ctx->nranks == 1) return rc;
    int worst = rc;
    const std::string mine = rc != SB_OK ? sb_last_error() : "";
    int rc2 = comm_allreduce_max_i32(ctx, &worst);
    if (rc2 != SB_OK) return rc2;
    if (rc != SB_OK) return sb_fail(rc, "%s", mine.c_str());
    if (worst != SB_OK) return sb_fail(worst, "%s: rejected on another rank", what);
    return SB_OK;
}

// O(nvec) host pass over the caller's pointer array: starts at 0, never decreases, ends at nnz.  The pipelined upload takes its
// copy extents from it, so it is checked before anything is copied or launched.
static int validate_indptr_host(const u64 *indptr, u64 nvec) {
    if (indptr[0] != 0) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: indptr is not monotone from 0");
    for (u64 i = 0; i < nvec; i++)
        if (indptr[i + 1] < indptr[i]) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: indptr is not monotone from 0 (at %llu)", (unsigned long long)i);
    return SB_OK;
}

static int upload_impl(sb_ctx *ctx, int major, uint32_t m, uint64_t n_local, const uint64_t *indptr, const HostEntries &he, sb_mat **out) {
    *out = nullptr;
    SB_ENTER(ctx);
    SB_TRY(agree_status(ctx, validate_indptr_host(indptr, major == SB_GENE_MAJOR ? (u64)m : n_local), "sb_upload"));
    trace_pool(ctx, "at upload start");
    SyncScope tr_total(ctx, "upload: whole call");
    u64 nvec = major == SB_GENE_MAJOR ? m : n_local;
    u64 nnz = indptr[nvec];
    std::unique_ptr<sb_mat> mt(new sb_mat());
    mt->ctx = ctx;
    mt->m = m;
    mt->n = n_local;
    mt->nnz = nnz;

    DevBuf<u64> d_ptr;
    DevEntries de;
    {
        SyncScope tr_a(ctx, "upload: staging allocations");
        SB_TRY(d_ptr.alloc(nvec + 1));
        SB_TRY(de.alloc(he, nnz, ctx->stream));
    }
    // large cell-major uploads take the pipelined path (copies overlapped with the layout build)
    const bool pipelined = major == SB_CELL_MAJOR && nnz >= ((u64)1 << 22) && n_local >= 8 * (u64)SB_MAX_PANEL_CELLS && TraceScope::level() != 1;
    if (pipelined) {
        SB_CUDA(cudaMemcpyAsync(d_ptr.p, indptr, (nvec + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        // private flags {pointer check, largest index}: the context scratch is also the staging buffer of the collectives
        // that set_global_shape / planes_select run on a sharded context
        DevBuf<int> flags;
        SB_TRY(flags.alloc(64));
        void *scr0 = flags.p;
        SB_CUDA(cudaMemsetAsync(scr0, 0, 256, ctx->stream));
        k_check_ptr<<<cdiv(nvec, 256), 256, 0, ctx->stream>>>(d_ptr.p, nvec, (int *)scr0);
        count_launch(ctx);
        mt->cm_ptr.swap(d_ptr);
        {
            SyncScope tr_b(ctx, "upload: cm allocation");
            SB_TRY(mt->cm.alloc(nnz));
        }
        SB_TRY(set_global_shape(mt.get()));
        {
            SyncScope tr_c(ctx, "upload: pipeline");
            SB_TRY(upload_pipelined(mt.get(), indptr, he, de, (u32 *)scr0 + 1));
        }
        trace_pool(ctx, "after pipeline");
        int hchk[2] = {0, 0};
        SB_CUDA(cudaMemcpyAsync(hchk, scr0, 8, cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        if (hchk[0]) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: indptr is not monotone from 0");
        if ((u64)(u32)hchk[1] >= (u64)m) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: index %u out of range %u", (u32)hchk[1], m);
        if (mt->gd == 0) SB_TRY(mat_ensure_full_gm(mt.get()));
        SB_TRY(finish_gather(mt.get()));
        *out = mt.release();
        return SB_OK;
    }
    SyncScope *tr_up = new SyncScope(ctx, "upload: H2D");
    prof_begin(ctx, PH_UPLOAD);
    SB_CUDA(cudaMemcpyAsync(d_ptr.p, indptr, (nvec + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    SB_TRY(copy_entries(he, de, 0, nnz, ctx->stream));
    prof_end(ctx, PH_UPLOAD);
    delete tr_up;
    ProfScope build_scope(ctx, PH_BUILD);
    SyncScope tr_build(ctx, "upload: build total");
    // interleave into {index, count} pairs; validation: pointers monotone, indices in range
    DevBuf<int> flags;
    SB_TRY(flags.alloc(64));
    void *scr = flags.p;
    SB_CUDA(cudaMemsetAsync(scr, 0, 256, ctx->stream));
    int *d_bad = (int *)scr;
    u32 *d_max = (u32 *)scr + 1;
    if (nvec) {
        k_check_ptr<<<cdiv(nvec, 256), 256, 0, ctx->stream>>>(d_ptr.p, nvec, d_bad);
        count_launch(ctx);
    }
    DevBuf<uint2> ent;
    SB_TRY(ent.alloc(nnz));
    SB_TRY(expand_entries(ctx, he, de, 0, nnz, ent.p, d_max, d_ptr.p, 0, nvec));
    int h[2] = {0, 0};
    SB_CUDA(cudaMemcpyAsync(h, scr, 8, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_TRY(packed_status(ctx, he, de));
    de.release();
    if (h[0]) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: indptr is not monotone from 0");
    u64 bound = major == SB_GENE_MAJOR ? n_local : (u64)m;
    if (nnz && (u64)(u32)h[1] >= bound) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: index %u out of range %llu", (u32)h[1], (unsigned long long)bound);

    SyncScope *tr_cm = new SyncScope(ctx, "upload: cell-major copy");
    if (major == SB_CELL_MAJOR) {
        mt->cm_ptr.swap(d_ptr);
        mt->cm.swap(ent);
    } else {
        // gene-major input: stable sort by cell gives the cell-major copy with ascending genes
        DevBuf<u32> keys;
        DevBuf<u64> payload;
        SB_TRY(keys.alloc(nnz));
        SB_TRY(payload.alloc(nnz));
        DevBuf<u32> hist;
        SB_TRY(hist.alloc(n_local + 1));
        SB_CUDA(cudaMemsetAsync(hist.p, 0, (n_local + 1) * sizeof(u32), ctx->stream));
        if (nnz) {
            k_make_keys<<<grid_for((u64)m * 32, 256, ctx, 16), 256, 0, ctx->stream>>>(d_ptr.p, ent.p, m, 1, m, 1, keys.p, payload.p);
            k_hist_u32<<<grid_for(nnz, 256, ctx, 16), 256, 0, ctx->stream>>>(keys.p, nnz, hist.p);
            count_launch(ctx); count_launch(ctx);
            SB_TRY(sort_pairs(ctx, keys, payload, nnz, bits_for(n_local ? n_local - 1 : 0)));
        }
        SB_TRY(mt->cm_ptr.alloc(n_local + 1));
        SB_TRY(exclusive_scan_u32_to_u64(ctx, hist.p, n_local, mt->cm_ptr.p));
        SB_TRY(mt->cm.alloc(nnz));
        if (nnz) {
            k_unpack_payload<<<grid_for(nnz, 256, ctx, 16), 256, 0, ctx->stream>>>(payload.p, mt->cm.p, nnz);
            count_launch(ctx);
        }
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    delete tr_cm;
    ent.release();
    SB_TRY(finish_matrix(mt.get()));
    *out = mt.release();
    return SB_OK;
}

extern "C" int sb_upload(sb_ctx *ctx, int major, uint32_t m, uint64_t n_local, const uint64_t *indptr, const uint32_t *idx,
                         const uint32_t *cnt, sb_mat **out) {
    if (!ctx || !out || !indptr) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: NULL argument");
    if (major != SB_GENE_MAJOR && major != SB_CELL_MAJOR) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: bad major %d", major);
    if (m > SB_GENE_MASK) return sb_fail(SB_ERR_UNSUPPORTED, "sb_upload: more than %u genes", SB_GENE_MASK);
    if (n_local > 0xFFFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "sb_upload: more than 2^32 cells per rank");
    const u64 nnz = indptr[major == SB_GENE_MAJOR ? (u64)m : n_local];
    if (nnz && (!idx || !cnt)) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload: NULL idx/cnt");
    HostEntries he;
    he.idx32 = idx;
    he.cnt32 = cnt;
    return upload_impl(ctx, major, m, n_local, indptr, he, out);
}

// Cell-major upload in the narrow host form: 3 bytes per entry over PCIe instead of 8 (the 11 GB of the 1.3M-cell matrix
// become 4.2 GB; the host -> device copy is the largest part of an end-to-end call).  Needs m <= 65536.
extern "C" int sb_upload_compact(sb_ctx *ctx, uint32_t m, uint64_t n_local, const uint64_t *indptr, const uint16_t *idx16,
                                 const uint8_t *cnt8, uint64_t n_big, const uint64_t *big_pos, const uint32_t *big_cnt, sb_mat **out) {
    if (!ctx || !out || !indptr) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_compact: NULL argument");
    if (m > 65536u) return sb_fail(SB_ERR_UNSUPPORTED, "sb_upload_compact: more than 65536 genes (use sb_upload)");
    if (n_local > 0xFFFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "sb_upload_compact: more than 2^32 cells per rank");
    const u64 nnz = indptr[n_local];
    if (nnz && (!idx16 || !cnt8)) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_compact: NULL idx16/cnt8");
    if (n_big && (!big_pos || !big_cnt)) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_compact: NULL side list");
    for (u64 i = 0; i < n_big; i++)
        if (big_pos[i] >= nnz || (i && big_pos[i] <= big_pos[i - 1]))
            return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_compact: side-list positions must be ascending and below nnz");
    HostEntries he;
    he.compact = true;
    he.idx16 = idx16;
    he.cnt8 = cnt8;
    he.n_big = n_big;
    he.big_pos = big_pos;
    he.big_cnt = big_cnt;
    return upload_impl(ctx, SB_CELL_MAJOR, m, n_local, indptr, he, out);
}

// Cell-major upload in the packed host form: one byte of gene delta and one nibble of count per entry (~1.55 B per entry over
// PCIe against 3 of the compact form and 8 of the plain one).  The decoder is k_expand_packed; sb_pack_csc_count / _fill
// (adaptive.cu) build the form on the host.
extern "C" int sb_upload_packed(sb_ctx *ctx, uint32_t m, uint64_t n_local, const uint64_t *indptr, const uint8_t *dgene, const uint8_t *cnt4,
                                uint64_t n_esc, const uint64_t *esc_pos, const uint32_t *esc_gene, uint64_t n_big, const uint64_t *big_pos,
                                const uint32_t *big_cnt, sb_mat **out) {
    if (!ctx || !out || !indptr) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_packed: NULL argument");
    if (m > SB_GENE_MASK) return sb_fail(SB_ERR_UNSUPPORTED, "sb_upload_packed: more than %u genes", SB_GENE_MASK);
    if (n_local > 0xFFFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "sb_upload_packed: more than 2^32 cells per rank");
    const u64 nnz = indptr[n_local];
    if (nnz && (!dgene || !cnt4)) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_packed: NULL dgene/cnt4");
    if ((n_big && (!big_pos || !big_cnt)) || (n_esc && (!esc_pos || !esc_gene))) return sb_fail(SB_ERR_INVALID_ARG, "sb_upload_packed: NULL side list");
    // the side lists are validated on the device (k_check_positions): millions of records
    HostEntries he;
    he.packed = true;
    he.dgene8 = dgene;
    he.cnt4 = cnt4;
    he.n_esc = n_esc;
    he.esc_pos = esc_pos;
    he.esc_gene = esc_gene;
    he.n_big = n_big;
    he.big_pos = big_pos;
    he.big_cnt = big_cnt;
    return upload_impl(ctx, SB_CELL_MAJOR, m, n_local, indptr, he, out);
}

// adopt device cell-major arrays (used by the synthetic generator and the selection routines)
int mat_from_device_cm(sb_ctx *ctx, u32 m, u64 n, DevBuf<u64> &cm_ptr, DevBuf<uint2> &cm, u64 nnz, sb_mat **out) {
    std::unique_ptr<sb_mat> mt(new sb_mat());
    mt->ctx = ctx;
    mt->m = m;
    mt->n = n;
    mt->nnz = nnz;
    mt->cm_ptr.swap(cm_ptr);
    mt->cm.swap(cm);
    SB_TRY(finish_matrix(mt.get()));
    *out = mt.release();
    return SB_OK;
}

extern "C" int sb_mat_shape(const sb_mat *mat, uint32_t *m, uint64_t *n_local, uint64_t *n_global, uint64_t *nnz_local) {
    if (!mat) return sb_fail(SB_ERR_INVALID_ARG, "sb_mat_shape: mat is NULL");
    if (m) *m = mat->m;
    if (n_local) *n_local = mat->n;
    if (n_global) *n_global = mat->n_global;
    if (nnz_local) *nnz_local = mat->nnz;
    return SB_OK;
}

extern "C" void sb_free_mat(sb_mat *mat) {
    if (!mat) return;
    cudaSetDevice(mat->ctx->device);
    sb_set_alloc_stream(mat->ctx->stream);
    cudaStreamSynchronize(mat->ctx->stream);
    delete mat;
}

extern "C" int sb_download(const sb_mat *mat, int major, uint64_t *indptr, uint32_t *idx, uint32_t *cnt) {
    if (!mat || !indptr) return sb_fail(SB_ERR_INVALID_ARG, "sb_download: NULL argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    u64 nnz = mat->nnz;
    DevBuf<u32> d_idx, d_cnt;
    SB_TRY(d_idx.alloc(nnz));
    SB_TRY(d_cnt.alloc(nnz));
    if (major == SB_CELL_MAJOR) {
        if (nnz) {
            k_split_entries<<<grid_for(nnz, 256, ctx, 16), 256, 0, ctx->stream>>>(mat->cm.p, nnz, d_idx.p, d_cnt.p);
            count_launch(ctx);
        }
        SB_CUDA(cudaMemcpyAsync(indptr, mat->cm_ptr.p, (mat->n + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    } else if (major == SB_GENE_MAJOR) {
        // stable sort of the cell-major stream by gene: cells ascending inside each gene
        DevBuf<u32> keys;
        DevBuf<u64> payload;
        DevBuf<u32> hist;
        DevBuf<u64> gptr;
        DevBuf<uint2> ent;
        SB_TRY(keys.alloc(nnz));
        SB_TRY(payload.alloc(nnz));
        SB_TRY(hist.alloc((size_t)mat->m + 1));
        SB_TRY(gptr.alloc((size_t)mat->m + 1));
        SB_TRY(ent.alloc(nnz));
        SB_CUDA(cudaMemsetAsync(hist.p, 0, ((size_t)mat->m + 1) * sizeof(u32), ctx->stream));
        if (nnz) {
            // mode 1 with vec = cell: key = ent.x (gene), payload = {cell, count}
            k_make_keys<<<grid_for(mat->n * 32, 256, ctx, 16), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, 1, mat->m, 1, keys.p, payload.p);
            k_hist_u32<<<grid_for(nnz, 256, ctx, 16), 256, 0, ctx->stream>>>(keys.p, nnz, hist.p);
            count_launch(ctx); count_launch(ctx);
            SB_TRY(sort_pairs(ctx, keys, payload, nnz, bits_for(mat->m ? mat->m - 1 : 0)));
            k_unpack_payload<<<grid_for(nnz, 256, ctx, 16), 256, 0, ctx->stream>>>(payload.p, ent.p, nnz);
            k_split_entries<<<grid_for(nnz, 256, ctx, 16), 256, 0, ctx->stream>>>(ent.p, nnz, d_idx.p, d_cnt.p);
            count_launch(ctx); count_launch(ctx);
        }
        SB_TRY(exclusive_scan_u32_to_u64(ctx, hist.p, mat->m, gptr.p));
        SB_CUDA(cudaMemcpyAsync(indptr, gptr.p, ((size_t)mat->m + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    } else {
        return sb_fail(SB_ERR_INVALID_ARG, "sb_download: bad major %d", major);
    }
    if (nnz && idx) SB_CUDA(cudaMemcpyAsync(idx, d_idx.p, nnz * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    if (nnz && cnt) SB_CUDA(cudaMemcpyAsync(cnt, d_cnt.p, nnz * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

// ---------------------------------------------------------------- integer reductions
int mat_cell_totals_dev(sb_mat *mat) {
    if (mat->have_cell_tot) return SB_OK;
    sb_ctx *ctx = mat->ctx;
    SB_TRY(mat->cell_tot.alloc(mat->n));
    if (mat->n) {
        ProfScope ps(ctx, PH_REDUCE);
        k_cell_totals<<<grid_for(mat->n * 32, 256, ctx, 16), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, mat->cell_tot.p);
        count_launch(ctx);
    }
    mat->have_cell_tot = true;
    return SB_OK;
}

extern "C" int sb_cell_totals(sb_mat *mat, uint32_t *out_n_local) {
    if (!mat || !out_n_local) return sb_fail(SB_ERR_INVALID_ARG, "sb_cell_totals: NULL argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    SB_TRY(mat_cell_totals_dev(mat));
    if (mat->n) SB_CUDA(cudaMemcpyAsync(out_n_local, mat->cell_tot.p, mat->n * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

int mat_gene_sums_dev(sb_mat *mat, int mode, const unsigned char *excl_cells, const unsigned char *excl_genes, u64 *d_out, bool allreduce) {
    sb_ctx *ctx = mat->ctx;
    SB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)mat->m * sizeof(u64), ctx->stream));
    if (mat->n && mat->nnz) {
        ProfScope ps(ctx, PH_REDUCE);
        k_gene_sums<<<grid_for(mat->n * 32, 256, ctx, 16), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, mode, excl_cells, excl_genes,
                                                                                  (unsigned long long *)d_out);
        count_launch(ctx);
    }
    if (allreduce) SB_TRY(comm_allreduce_u64(ctx, d_out, mat->m));
    return SB_OK;
}

static int gene_sums_host(sb_mat *mat, int mode, uint64_t *out_m) {
    if (!mat || !out_m) return sb_fail(SB_ERR_INVALID_ARG, "gene sums: NULL argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    DevBuf<u64> d;
    SB_TRY(d.alloc(mat->m));
    SB_TRY(mat_gene_sums_dev(mat, mode, nullptr, nullptr, d.p, true));
    if (mat->m) SB_CUDA(cudaMemcpyAsync(out_m, d.p, (size_t)mat->m * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

extern "C" int sb_gene_totals(sb_mat *mat, int square, uint64_t *out_m) { return gene_sums_host(mat, square ? 1 : 0, out_m); }
extern "C" int sb_gene_nnz(sb_mat *mat, uint64_t *out_m) { return gene_sums_host(mat, 2, out_m); }

// K3: median of the cell totals over all ranks (scan-rs/src/stats.rs:13-38)
int mat_median_total(sb_mat *mat, u32 *median, int *nonempty) {
    sb_ctx *ctx = mat->ctx;
    SB_TRY(mat_cell_totals_dev(mat));
    u64 ng = mat->n_global;
    *nonempty = ng > 0;
    *median = 0;
    if (ng == 0) return SB_OK;
    ProfScope ps(ctx, PH_REDUCE);
    DevBuf<u32> all, sorted;
    SB_TRY(all.alloc(ng));
    SB_TRY(sorted.alloc(ng));
    if (ctx->nranks == 1) {
        SB_CUDA(cudaMemcpyAsync(all.p, mat->cell_tot.p, ng * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        std::vector<u64> counts;
        SB_TRY(comm_allgather_u64_host(ctx, mat->n, counts));
        SB_NCCL(ncclGroupStart());
        u64 off = 0;
        for (int r = 0; r < ctx->nranks; r++) {
            if (counts[r]) SB_NCCL(ncclBroadcast(mat->cell_tot.p, all.p + off, counts[r], ncclUint32, r, ctx->comm, ctx->stream));
            off += counts[r];
        }
        SB_NCCL(ncclGroupEnd());
        count_launch(ctx, false);
    }
    size_t tmp_bytes = 0;
    SB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tmp_bytes, all.p, sorted.p, (unsigned long long)ng, 0, 32, ctx->stream));
    DevBuf<char> tmp;
    SB_TRY(tmp.alloc(tmp_bytes));
    SB_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, tmp_bytes, all.p, sorted.p, (unsigned long long)ng, 0, 32, ctx->stream));
    count_launch(ctx, false);
    u32 h[2] = {0, 0};
    if (ng % 2 == 0) {
        SB_CUDA(cudaMemcpyAsync(h, sorted.p + (ng / 2 - 1), 2 * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        *median = (u32)(h[0] + h[1]) / 2u;  // u32 wrapping add, integer divide (stats.rs:32)
    } else {
        SB_CUDA(cudaMemcpyAsync(h, sorted.p + ng / 2, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        *median = h[0];
    }
    return SB_OK;
}

extern "C" int sb_median_cell_total(sb_mat *mat, uint32_t *median, int *nonempty) {
    if (!mat || !median || !nonempty) return sb_fail(SB_ERR_INVALID_ARG, "sb_median_cell_total: NULL argument");
    SB_ENTER(mat->ctx);
    return mat_median_total(mat, median, nonempty);
}

// ---------------------------------------------------------------- selection
// general form of the row selection: gene g is wanted at positions inv_list[inv_ptr[g] .. inv_ptr[g+1]) of the output
__global__ void k_select_rows_multi(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, const u32 *__restrict__ inv_ptr,
                                    const u32 *__restrict__ inv_list, const u64 *__restrict__ new_ptr, u32 *__restrict__ counts,
                                    u32 *__restrict__ out_gene, u32 *__restrict__ out_cnt) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        const u64 s = ptr[c], e = ptr[c + 1];
        const u64 wpos = new_ptr ? new_ptr[c] : 0;
        u32 total = 0;
        for (u64 k0 = s; k0 < e; k0 += 32) {
            const u64 k = k0 + lane;
            const uint2 z = k < e ? cm[k] : make_uint2(0, 0);
            const u32 a = k < e ? inv_ptr[z.x] : 0, b = k < e ? inv_ptr[z.x + 1] : 0;
            const u32 mine = b - a;
            u32 incl = mine;  // inclusive warp scan of the copies each lane emits
            for (int o = 1; o < 32; o <<= 1) {
                const u32 t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (out_gene)
                for (u32 i = 0; i < mine; i++) {
                    out_gene[wpos + total + incl - mine + i] = inv_list[a + i];
                    out_cnt[wpos + total + incl - mine + i] = z.y;
                }
            total += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (counts && lane == 0) counts[c] = total;
    }
}

__global__ void k_zip_entries(const u32 *__restrict__ gene, const u32 *__restrict__ cnt, u64 nnz, uint2 *__restrict__ out) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (u64)gridDim.x * blockDim.x) out[i] = make_uint2(gene[i], cnt[i]);
}

// select_rows (sqz/src/mat.rs:1040-1071): the output's row j is a clone of row rows[j] -- any order, duplicates allowed.
static int select_rows_dev(sb_mat *mat, const u32 *h_rows, u32 count, sb_mat **out) {
    sb_ctx *ctx = mat->ctx;
    bool ascending = true;
    for (u32 j = 0; j < count; j++) {
        if (h_rows[j] >= mat->m) return sb_fail(SB_ERR_INVALID_ARG, "select_rows: row %u out of range", h_rows[j]);
        if (j && h_rows[j] <= h_rows[j - 1]) ascending = false;
    }
    DevBuf<u32> d_counts;
    DevBuf<u64> new_ptr;
    DevBuf<uint2> new_cm;
    SB_TRY(d_counts.alloc(mat->n));
    SB_TRY(new_ptr.alloc(mat->n + 1));
    int grid = grid_for(mat->n * 32, 256, ctx, 16);
    u64 new_nnz = 0;
    if (ascending) {  // one output position per gene and the cells' entries stay in ascending order
        std::vector<u32> map(mat->m, 0xFFFFFFFFu);
        for (u32 j = 0; j < count; j++) map[h_rows[j]] = j;
        DevBuf<u32> d_map;
        SB_TRY(d_map.alloc(mat->m));
        if (mat->m) SB_CUDA(cudaMemcpyAsync(d_map.p, map.data(), (size_t)mat->m * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        if (mat->n) {
            k_select_rows<<<grid, 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, d_map.p, nullptr, d_counts.p, nullptr);
            count_launch(ctx);
        }
        SB_TRY(exclusive_scan_u32_to_u64(ctx, d_counts.p, mat->n, new_ptr.p));
        SB_CUDA(cudaMemcpyAsync(&new_nnz, new_ptr.p + mat->n, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));  // also: `map` is a host temporary
        SB_TRY(new_cm.alloc(new_nnz));
        if (mat->n) {
            k_select_rows<<<grid, 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, d_map.p, new_ptr.p, nullptr, new_cm.p);
            count_launch(ctx);
        }
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        return mat_from_device_cm(ctx, count, mat->n, new_ptr, new_cm, new_nnz, out);
    }
    // general order: every wanted copy of a gene is emitted, then each cell's entries are sorted by their new row
    std::vector<u32> inv_ptr((size_t)mat->m + 1, 0), inv_list(count ? count : 1, 0);
    for (u32 j = 0; j < count; j++) inv_ptr[h_rows[j] + 1]++;
    for (u32 g = 0; g < mat->m; g++) inv_ptr[g + 1] += inv_ptr[g];
    {
        std::vector<u32> fill(inv_ptr.begin(), inv_ptr.end() - 1);
        for (u32 j = 0; j < count; j++) inv_list[fill[h_rows[j]]++] = j;
    }
    DevBuf<u32> d_iptr, d_ilist, g_in, c_in, g_out, c_out;
    SB_TRY(d_iptr.alloc(inv_ptr.size()));
    SB_TRY(d_ilist.alloc(inv_list.size()));
    SB_CUDA(cudaMemcpyAsync(d_iptr.p, inv_ptr.data(), inv_ptr.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(d_ilist.p, inv_list.data(), inv_list.size() * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    if (mat->n) {
        k_select_rows_multi<<<grid, 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, d_iptr.p, d_ilist.p, nullptr, d_counts.p, nullptr, nullptr);
        count_launch(ctx);
    }
    SB_TRY(exclusive_scan_u32_to_u64(ctx, d_counts.p, mat->n, new_ptr.p));
    SB_CUDA(cudaMemcpyAsync(&new_nnz, new_ptr.p + mat->n, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_TRY(g_in.alloc(new_nnz));
    SB_TRY(c_in.alloc(new_nnz));
    SB_TRY(g_out.alloc(new_nnz));
    SB_TRY(c_out.alloc(new_nnz));
    SB_TRY(new_cm.alloc(new_nnz));
    if (mat->n && new_nnz) {
        k_select_rows_multi<<<grid, 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, d_iptr.p, d_ilist.p, new_ptr.p, nullptr, g_in.p, c_in.p);
        count_launch(ctx);
        if (new_nnz > 0x7FFFFFFFull) return sb_fail(SB_ERR_UNSUPPORTED, "select_rows: more than 2^31 entries in a reordering selection");
        size_t tmp_bytes = 0;
        const int end_bit = bits_for(count ? count - 1 : 0);
        SB_CUDA(cub::DeviceSegmentedRadixSort::SortPairs(nullptr, tmp_bytes, g_in.p, g_out.p, c_in.p, c_out.p, (int)new_nnz, (int)mat->n, new_ptr.p,
                                                         new_ptr.p + 1, 0, end_bit, ctx->stream));
        DevBuf<char> tmp;
        SB_TRY(tmp.alloc(tmp_bytes));
        SB_CUDA(cub::DeviceSegmentedRadixSort::SortPairs(tmp.p, tmp_bytes, g_in.p, g_out.p, c_in.p, c_out.p, (int)new_nnz, (int)mat->n, new_ptr.p,
                                                         new_ptr.p + 1, 0, end_bit, ctx->stream));
        count_launch(ctx, false);
        k_zip_entries<<<grid_for(new_nnz, 256, ctx, 16), 256, 0, ctx->stream>>>(g_out.p, c_out.p, new_nnz, new_cm.p);
        count_launch(ctx);
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return mat_from_device_cm(ctx, count, mat->n, new_ptr, new_cm, new_nnz, out);
}

static int select_cols_dev(sb_mat *mat, const u64 *h_cols, u64 count, sb_mat **out) {
    sb_ctx *ctx = mat->ctx;
    for (u64 j = 0; j < count; j++)
        if (h_cols[j] >= mat->n) return sb_fail(SB_ERR_INVALID_ARG, "select_cols: column %llu out of range", (unsigned long long)h_cols[j]);
    DevBuf<u64> d_cols, new_ptr;
    DevBuf<u32> d_len;
    SB_TRY(d_cols.alloc(count));
    SB_TRY(d_len.alloc(count));
    SB_TRY(new_ptr.alloc(count + 1));
    if (count) {
        SB_CUDA(cudaMemcpyAsync(d_cols.p, h_cols, count * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        k_gather_len<<<cdiv(count, 256), 256, 0, ctx->stream>>>(mat->cm_ptr.p, d_cols.p, count, d_len.p);
        count_launch(ctx);
    }
    SB_TRY(exclusive_scan_u32_to_u64(ctx, d_len.p, count, new_ptr.p));
    u64 new_nnz = 0;
    SB_CUDA(cudaMemcpyAsync(&new_nnz, new_ptr.p + count, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    DevBuf<uint2> new_cm;
    SB_TRY(new_cm.alloc(new_nnz));
    if (count) {
        k_select_cols<<<grid_for(count * 32, 256, ctx, 16), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, d_cols.p, count, new_ptr.p, new_cm.p);
        count_launch(ctx);
    }
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return mat_from_device_cm(ctx, mat->m, count, new_ptr, new_cm, new_nnz, out);
}

extern "C" int sb_select_rows(sb_mat *mat, const uint32_t *rows, uint32_t count, sb_mat **out) {
    if (!mat || !out || (count && !rows)) return sb_fail(SB_ERR_INVALID_ARG, "sb_select_rows: NULL argument");
    SB_ENTER(mat->ctx);
    *out = nullptr;
    return select_rows_dev(mat, rows, count, out);
}

extern "C" int sb_select_cols(sb_mat *mat, const uint64_t *cols, uint64_t count, sb_mat **out) {
    if (!mat || !out || (count && !cols)) return sb_fail(SB_ERR_INVALID_ARG, "sb_select_cols: NULL argument");
    SB_ENTER(mat->ctx);
    *out = nullptr;
    return select_cols_dev(mat, cols, count, out);
}

// K4: partition_on_thresholds (sqz/src/mat.rs:772-889)
extern "C" int sb_partition(sb_mat *mat, int has_row_thr, double row_thr, int has_col_thr, double col_thr, sb_mat **kept,
                            sb_mat **residual, uint64_t *rows_out, uint64_t *n_rows_out, uint64_t *cols_out, uint64_t *n_cols_out) {
    if (!mat) return sb_fail(SB_ERR_INVALID_ARG, "sb_partition: mat is NULL");
    sb_ctx *ctx = mat->ctx;
    // Sharded contexts (SURVEY 8e): a cell belongs to one rank, so the column sums and the column verdicts stay local; the row
    // (gene) sums are all-reduced every round (exact u64) and so is the "something changed" flag -- every rank runs the same
    // number of rounds and ends with the same row set.  cols_out are LOCAL cell indices.
    SB_ENTER(ctx);
    if (kept) *kept = nullptr;
    if (residual) *residual = nullptr;
    DevBuf<unsigned char> ex_rows, ex_cols;
    DevBuf<u64> sums;
    SB_TRY(ex_rows.alloc(mat->m));
    SB_TRY(ex_cols.alloc(mat->n));
    SB_TRY(sums.alloc(std::max<u64>(mat->m, mat->n)));
    SB_CUDA(cudaMemsetAsync(ex_rows.p, 0, mat->m ? mat->m : 1, ctx->stream));
    SB_CUDA(cudaMemsetAsync(ex_cols.p, 0, mat->n ? mat->n : 1, ctx->stream));
    DevBuf<int> upd_flag;  // private: the context scratch is the staging buffer of the collectives below
    SB_TRY(upd_flag.alloc(1));
    int *d_upd = upd_flag.p;
    for (;;) {
        SB_CUDA(cudaMemsetAsync(d_upd, 0, sizeof(int), ctx->stream));
        if (has_col_thr && mat->n) {  // mat.rs:783-790
            k_cell_sums_masked<<<grid_for(mat->n * 32, 256, ctx, 16), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, ex_cols.p, ex_rows.p,
                                                                                            (unsigned long long *)sums.p);
            k_apply_threshold<<<cdiv(mat->n, 256), 256, 0, ctx->stream>>>((unsigned long long *)sums.p, mat->n, col_thr, ex_cols.p, d_upd);
            count_launch(ctx); count_launch(ctx);
        }
        if (has_row_thr && mat->m) {  // mat.rs:791-798
            SB_TRY(mat_gene_sums_dev(mat, 0, ex_cols.p, ex_rows.p, sums.p, ctx->nranks > 1));
            k_apply_threshold<<<cdiv(mat->m, 256), 256, 0, ctx->stream>>>((unsigned long long *)sums.p, mat->m, row_thr, ex_rows.p, d_upd);
            count_launch(ctx);
        }
        int upd = 0;
        SB_CUDA(cudaMemcpyAsync(&upd, d_upd, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        if (ctx->nranks > 1) SB_TRY(comm_allreduce_max_i32(ctx, &upd));
        if (!upd) break;
    }
    std::vector<unsigned char> hr(mat->m), hc(mat->n);
    if (mat->m) SB_CUDA(cudaMemcpyAsync(hr.data(), ex_rows.p, mat->m, cudaMemcpyDeviceToHost, ctx->stream));
    if (mat->n) SB_CUDA(cudaMemcpyAsync(hc.data(), ex_cols.p, mat->n, cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    std::vector<u32> sel_rows;
    std::vector<u64> sel_cols, exc_cols;
    for (u32 r = 0; r < mat->m; r++)
        if (!hr[r]) sel_rows.push_back(r);
    for (u64 c = 0; c < mat->n; c++) (hc[c] ? exc_cols : sel_cols).push_back(c);
    if (rows_out)
        for (size_t i = 0; i < sel_rows.size(); i++) rows_out[i] = sel_rows[i];
    if (n_rows_out) *n_rows_out = sel_rows.size();
    if (cols_out)
        for (size_t i = 0; i < sel_cols.size(); i++) cols_out[i] = sel_cols[i];
    if (n_cols_out) *n_cols_out = sel_cols.size();
    if (kept || residual) {
        sb_mat *rows_kept = nullptr;
        SB_TRY(select_rows_dev(mat, sel_rows.data(), (u32)sel_rows.size(), &rows_kept));
        int rc = SB_OK;
        if (kept) rc = select_cols_dev(rows_kept, sel_cols.data(), sel_cols.size(), kept);
        if (rc == SB_OK && residual) rc = select_cols_dev(rows_kept, exc_cols.data(), exc_cols.size(), residual);
        sb_free_mat(rows_kept);
        if (rc != SB_OK) {
            if (kept && *kept) { sb_free_mat(*kept); *kept = nullptr; }
            return rc;
        }
    }
    return SB_OK;
}

// K6 + host top-N (builder-defined, SURVEY 8c): exact u64 sums -> f64 dispersion -> stable top-N
extern "C" int sb_hvg_select(sb_mat *mat, uint32_t n_top, uint32_t *out_idx, uint32_t *out_count) {
    if (!mat || !out_idx || !out_count) return sb_fail(SB_ERR_INVALID_ARG, "sb_hvg_select: NULL argument");
    std::vector<u64> s1(mat->m), s2(mat->m);
    SB_TRY(sb_gene_totals(mat, 0, s1.data()));
    SB_TRY(sb_gene_totals(mat, 1, s2.data()));
    double n = (double)mat->n_global;
    std::vector<double> disp(mat->m);
    for (u32 g = 0; g < mat->m; g++) {
        double mean = (double)s1[g] / n;
        double var = (double)s2[g] / n - mean * mean;
        disp[g] = mean > 0.0 ? var / mean : 0.0;
    }
    std::vector<u32> order(mat->m);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](u32 a, u32 b) { return disp[a] > disp[b]; });
    u32 cnt = std::min<u32>(n_top, mat->m);
    std::vector<u32> top(order.begin(), order.begin() + cnt);
    std::sort(top.begin(), top.end());
    for (u32 i = 0; i < cnt; i++) out_idx[i] = top[i];
    *out_count = cnt;
    return SB_OK;
}
