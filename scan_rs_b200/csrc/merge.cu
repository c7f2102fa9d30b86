// merge.cu -- merging of over-split clusters by differential expression (Cell Ranger's MERGE_CLUSTERS step; scan-rs's linkage.rs
// and merge_clusters.rs).  The rule is stated beside sb_merge_clusters in include/scanb200.h and restated by
// oracle/merge_clusters.py.
//
//   gene sums   group_gene_sums (diff_exp.cu's k_group_sums + one u64 all-reduce) once for the input groups; a merge adds row b into
//               row a on the device (exact in u64), so the loop never reads the matrix again
//   per round   cell ids sorted by current cluster (sort_pairs is a stable radix sort: ascending cell order inside a cluster), then
//               k_group_seq_sums sums the score columns and the size factors of every cluster in that order (a thread per
//               (cluster, column)), so centroid and s bits depend on neither the grid nor the world size; complete linkage of the
//               centroids on the host (linkage.h); the sibling leaf pairs go through sb_sseq_pairs' test path (sseq_pair_tests)
// Sharded contexts: labels, size factors and score rows are gathered in global cell order and every rank runs the same loop; the
// gene sums are all-reduced and the tests stay sharded inside the test stage.
#include <cmath>
#include <numeric>

#include "common.cuh"
#include "linkage.h"

#define MG_MAX_DIM 128  // knn.cu's limit

static int mg_grid(sb_ctx *ctx, u64 items, int per_block) {
    return (int)std::max<u64>(1, std::min<u64>((items + per_block - 1) / per_block, (u64)ctx->sm_count * 16));
}

// sort keys: the current cluster of every cell (cur[] maps input groups to current clusters), values: the cell id
__global__ void k_mg_keys(const u32 *__restrict__ lab, const u32 *__restrict__ cur, u64 n, u64 *__restrict__ keys, u64 *__restrict__ vals) {
    for (u64 c = (u64)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (u64)gridDim.x * blockDim.x) {
        keys[c] = cur[lab[c]];
        vals[c] = c;
    }
}

// a thread per (group, column): out[g * ncol + col] = sum of X[cell * ld + col] over cells order[off[g] .. off[g + 1]), in that order
__global__ void k_group_seq_sums(const double *__restrict__ X, u32 ld, u32 ncol, const u64 *__restrict__ order, const u64 *__restrict__ off, u32 ngroups,
                                 double *__restrict__ out) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < (u64)ngroups * ncol; t += (u64)gridDim.x * blockDim.x) {
        const u64 g = t / ncol, col = t % ncol, e = off[g + 1];
        double s = 0.0;
#pragma unroll 8
        for (u64 i = off[g]; i < e; i++) s = __dadd_rn(s, X[order[i] * ld + col]);
        out[t] = s;
    }
}

// acc row mv[j].x += row mv[j].y (the rows of one round are distinct)
__global__ void k_mg_add_rows(u64 *__restrict__ acc, u32 m, const uint2 *__restrict__ mv, u32 nmv) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < (u64)nmv * m; t += (u64)gridDim.x * blockDim.x) {
        const uint2 r = mv[t / m];
        acc[(u64)r.x * m + t % m] += acc[(u64)r.y * m + t % m];
    }
}

__global__ void k_mg_finite(const double *__restrict__ X, u64 count, int *__restrict__ bad) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (u64)gridDim.x * blockDim.x)
        if (!isfinite(X[i])) atomicOr(bad, 1);
}

extern "C" int sb_linkage_complete(const double *points, uint32_t n, uint32_t dim, double *Z) {
    if ((!points && n) || (!Z && n > 1) || n == 0 || dim == 0) return sb_fail(SB_ERR_INVALID_ARG, "sb_linkage_complete: bad argument (n >= 1, dim >= 1)");
    if (n > SB_LINKAGE_MAX_POINTS) return sb_fail(SB_ERR_UNSUPPORTED, "sb_linkage_complete: n must be <= %d", SB_LINKAGE_MAX_POINTS);
    for (u64 i = 0; i < (u64)n * dim; i++)
        if (!std::isfinite(points[i])) return sb_fail(SB_ERR_INVALID_ARG, "sb_linkage_complete: coordinate %llu is not finite", (unsigned long long)i);
    if (!linkage_complete_host(points, n, dim, Z)) return sb_fail(SB_ERR_INVALID_ARG, "sb_linkage_complete: a distance is not finite");
    return SB_OK;
}

extern "C" int sb_merge_clusters(sb_mat *mat, const sb_sseq_params *params, const double *scores, uint32_t dim, const uint32_t *labels,
                                 uint32_t n_groups, const sb_merge_opts *opts, uint32_t *labels_out, sb_merge_info *info) {
    static const char *fn = "sb_merge_clusters";
    if (!mat) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn);
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    const sb_merge_opts o = opts ? *opts : sb_merge_opts{0.05, 1, 0, 900};
    int rc = (!info || (mat->n && (!scores || !labels || !labels_out))) ? sb_fail(SB_ERR_INVALID_ARG, "%s: NULL argument", fn) : SB_OK;
    if (rc == SB_OK && !(o.adj_p_threshold > 0.0 && o.adj_p_threshold <= 1.0)) rc = sb_fail(SB_ERR_INVALID_ARG, "%s: adj_p_threshold must be in (0, 1]", fn);
    if (rc == SB_OK && (dim == 0 || dim > MG_MAX_DIM)) rc = sb_fail(SB_ERR_INVALID_ARG, "%s: dim must be 1..%d", fn, MG_MAX_DIM);
    if (rc == SB_OK && n_groups == 0) rc = sb_fail(SB_ERR_INVALID_ARG, "%s: n_groups must be >= 1", fn);
    if (rc == SB_OK && n_groups > SB_LINKAGE_MAX_POINTS) rc = sb_fail(SB_ERR_UNSUPPORTED, "%s: n_groups must be <= %d", fn, SB_LINKAGE_MAX_POINTS);
    if (rc == SB_OK) rc = sseq_check_params(mat, params, fn);
    for (u64 c = 0; c < mat->n && rc == SB_OK; c++)
        if (labels[c] >= n_groups)
            rc = sb_fail(SB_ERR_INVALID_ARG, "%s: label %u of cell %llu is not below n_groups = %u", fn, labels[c], (unsigned long long)(mat->cell_offset + c),
                         n_groups);
    SB_TRY(agree_status(ctx, rc, fn));
    const u32 m = mat->m;

    // labels, size factors and score rows of all cells in global cell order
    std::vector<u64> counts, shape;
    SB_TRY(comm_allgather_u64_host(ctx, mat->n, counts));
    SB_TRY(comm_allgather_u64_host(ctx, dim, shape));
    u64 n = 0, maxr = 0, off = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        if (shape[r] != dim) return sb_fail(SB_ERR_INVALID_ARG, "%s: dim differs between ranks (rank %d)", fn, r);
        if (r < ctx->rank) off += counts[r];
        n += counts[r];
        maxr = std::max(maxr, counts[r]);
    }
    std::vector<u32> lab(n);
    std::vector<double> sf;
    DevBuf<double> dX, dS;
    DevBuf<u32> dL;
    std::vector<u64> size(n_groups, 0);
    {
        TraceScope tr(ctx, "merge: cell gathers");
        std::vector<double> lab_l(mat->n), labd;
        for (u64 c = 0; c < mat->n; c++) lab_l[c] = (double)labels[c];
        SB_TRY(gather_cells(ctx, lab_l, labd));
        SB_TRY(gather_cells(ctx, std::vector<double>(params->size_factors, params->size_factors + mat->n), sf));
        for (u64 c = 0; c < n; c++) {
            lab[c] = (u32)labd[c];
            size[lab[c]]++;
        }
        SB_TRY(dX.alloc(n * dim));
        SB_TRY(dS.alloc(n));
        SB_TRY(dL.alloc(n));
        if (ctx->nranks == 1) {
            if (n) SB_CUDA(cudaMemcpyAsync(dX.p, scores, n * dim * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        } else {
            SB_TRY(um_gather_rows(ctx, scores, mat->n, 2 * (u64)dim, counts, maxr, (u32 *)dX.p));
        }
        if (n) {
            SB_CUDA(cudaMemcpyAsync(dS.p, sf.data(), n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
            SB_CUDA(cudaMemcpyAsync(dL.p, lab.data(), n * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        }
        DevBuf<int> bad;
        SB_TRY(bad.alloc(1));
        SB_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), ctx->stream));
        if (n) {
            k_mg_finite<<<mg_grid(ctx, n * dim, 256), 256, 0, ctx->stream>>>(dX.p, n * dim, bad.p);
            count_launch(ctx);
            SB_CUDA(cudaGetLastError());
        }
        int hbad = 0;
        SB_CUDA(cudaMemcpyAsync(&hbad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        rc = hbad ? sb_fail(SB_ERR_INVALID_ARG, "%s: a score is not finite", fn) : SB_OK;
        for (u32 g = 0; g < n_groups && rc == SB_OK; g++)
            if (!size[g]) rc = sb_fail(SB_ERR_INVALID_ARG, "%s: group %u is empty", fn, g);
        SB_TRY(agree_status(ctx, rc, fn));
    }

    // current clusters: cur[input group] -> cluster id, rep[cluster] -> its row of the gene sums, csize[cluster]
    std::vector<u32> cur(n_groups), rep(n_groups);
    std::iota(cur.begin(), cur.end(), 0u);
    std::iota(rep.begin(), rep.end(), 0u);
    std::vector<u64> csize = size;
    u32 K = n_groups;
    sb_merge_info inf{n_groups, 0, 0, 0};
    DevBuf<u64> acc;
    if (K > 1) {
        TraceScope tr(ctx, "merge: group sums");
        SB_TRY(group_gene_sums(mat, dL.p + off, n_groups, acc));
    }
    DevBuf<u32> dcur;
    DevBuf<u64> keys, vals, doff;
    DevBuf<double> dsum, ds;
    SB_TRY(dcur.alloc(n_groups));
    SB_TRY(doff.alloc(n_groups + 1));
    SB_TRY(dsum.alloc((u64)n_groups * dim));
    SB_TRY(ds.alloc(n_groups));
    while (K > 1) {
        inf.n_rounds++;
        std::vector<double> cent((u64)K * dim), s(K);
        {
            TraceScope tr(ctx, "merge: centroids");
            SB_TRY(keys.alloc(n));
            SB_TRY(vals.alloc(n));
            std::vector<u64> ofs(K + 1, 0);
            for (u32 k = 0; k < K; k++) ofs[k + 1] = ofs[k] + csize[k];
            SB_CUDA(cudaMemcpyAsync(dcur.p, cur.data(), n_groups * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
            SB_CUDA(cudaMemcpyAsync(doff.p, ofs.data(), (K + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
            k_mg_keys<<<mg_grid(ctx, n, 256), 256, 0, ctx->stream>>>(dL.p, dcur.p, n, keys.p, vals.p);
            count_launch(ctx);
            SB_TRY(sort_pairs(ctx, keys, vals, n));
            k_group_seq_sums<<<mg_grid(ctx, (u64)K * dim, 128), 128, 0, ctx->stream>>>(dX.p, dim, dim, vals.p, doff.p, K, dsum.p);
            k_group_seq_sums<<<mg_grid(ctx, K, 128), 128, 0, ctx->stream>>>(dS.p, 1, 1, vals.p, doff.p, K, ds.p);
            count_launch(ctx);
            count_launch(ctx);
            SB_CUDA(cudaGetLastError());
            SB_CUDA(cudaMemcpyAsync(cent.data(), dsum.p, (u64)K * dim * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            SB_CUDA(cudaMemcpyAsync(s.data(), ds.p, K * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            SB_CUDA(cudaStreamSynchronize(ctx->stream));
            for (u32 k = 0; k < K; k++)
                for (u32 c = 0; c < dim; c++) cent[(u64)k * dim + c] /= (double)csize[k];
        }
        std::vector<u32> rows, pa, pb;
        std::vector<double> s_in, s_out;
        {
            TraceScope tr(ctx, "merge: linkage");
            std::vector<double> Z((u64)(K - 1) * 4);
            if (!linkage_complete_host(cent.data(), K, dim, Z.data())) return sb_fail(SB_ERR_INVALID_ARG, "%s: a centroid distance is not finite", fn);
            for (u32 i = 0; i + 1 < K; i++) {
                const double a = Z[(u64)i * 4], b = Z[(u64)i * 4 + 1];
                if (a < K && b < K) {
                    pa.push_back((u32)a);
                    pb.push_back((u32)b);
                    rows.push_back(rep[(u32)a]);
                    rows.push_back(rep[(u32)b]);
                    s_in.push_back(s[(u32)a]);
                    s_out.push_back(s[(u32)b]);
                }
            }
        }
        const u32 np = (u32)pa.size();
        inf.pairs_tested += np;
        const u64 tot = (u64)np * m;
        std::vector<u64> h_in(tot), h_out(tot);
        std::vector<double> nm_in(tot), nm_out(tot), pv(tot), q(tot), lfc(tot);
        sb_diff_exp_out de{h_in.data(), h_out.data(), nm_in.data(), nm_out.data(), pv.data(), q.data(), lfc.data()};
        {
            TraceScope tr(ctx, "merge: tests");
            SB_TRY(sseq_pair_tests(mat, params, acc.p, rows, s_in, s_out, o.big_count, &de));
        }
        TraceScope tr(ctx, "merge: host tail");
        std::vector<uint2> mv;
        std::vector<u32> into(K);
        std::iota(into.begin(), into.end(), 0u);
        for (u32 j = 0; j < np; j++) {
            u64 de_genes = 0;
            for (u32 g = 0; g < m; g++) de_genes += q[(u64)j * m + g] < o.adj_p_threshold;
            if (de_genes < o.min_de_genes) {
                into[pb[j]] = pa[j];
                mv.push_back(make_uint2(rep[pa[j]], rep[pb[j]]));
            }
        }
        if (mv.empty()) break;
        inf.pairs_merged += mv.size();
        DevBuf<uint2> dmv;
        SB_TRY(dmv.alloc(mv.size()));
        SB_CUDA(cudaMemcpyAsync(dmv.p, mv.data(), mv.size() * sizeof(uint2), cudaMemcpyHostToDevice, ctx->stream));
        k_mg_add_rows<<<mg_grid(ctx, (u64)mv.size() * m, 256), 256, 0, ctx->stream>>>(acc.p, m, dmv.p, (u32)mv.size());
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        // renumber the survivors in ascending old id
        std::vector<u32> nid(K, 0), rep2;
        std::vector<u64> csize2;
        for (u32 k = 0; k < K; k++)
            if (into[k] == k) {
                nid[k] = (u32)rep2.size();
                rep2.push_back(rep[k]);
                csize2.push_back(0);
            }
        for (u32 k = 0; k < K; k++) csize2[nid[into[k]]] += csize[k];
        for (u32 g = 0; g < n_groups; g++) cur[g] = nid[into[cur[g]]];
        rep.swap(rep2);
        csize.swap(csize2);
        K = (u32)rep.size();
    }
    // final labels: by size, descending, ties to the smallest global cell index
    TraceScope tr(ctx, "merge: host tail");
    std::vector<u64> first(K, ~0ull);
    for (u64 c = 0; c < n; c++) first[cur[lab[c]]] = std::min(first[cur[lab[c]]], c);
    std::vector<u32> ids(K), rank(K);
    std::iota(ids.begin(), ids.end(), 0u);
    std::sort(ids.begin(), ids.end(), [&](u32 x, u32 y) { return csize[x] != csize[y] ? csize[x] > csize[y] : first[x] < first[y]; });
    for (u32 r = 0; r < K; r++) rank[ids[r]] = r;
    for (u64 c = 0; c < mat->n; c++) labels_out[c] = rank[cur[labels[c]]];
    inf.n_clusters = K;
    *info = inf;
    return SB_OK;
}
