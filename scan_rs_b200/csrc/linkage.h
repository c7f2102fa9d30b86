// linkage.h -- complete-linkage hierarchical clustering of a few thousand points on the host: the NN-chain algorithm of scan-rs's
// linkage.rs (and of scipy's nn_chain), used by merge.cu on the cluster centroids.  Header-only, no CUDA, no context.
//
// Rule (stated again beside sb_linkage_complete in include/scanb200.h):
//   d(i, j)   = sqrt(sum_c (x_j,c - x_i,c)^2), summed in coordinate order with one rounding per operation (knn.cu's expression);
//               between clusters the largest point distance (Lance-Williams: d(k, i u j) = max(d(k, i), d(k, j))).
//   chain     starts at the lowest active slot; the next element is the active slot nearest to the chain's top, where the element
//               below the top wins a tie with it and otherwise the lowest slot wins; two mutual nearest neighbours x < y merge at
//               height d(x, y) and the merged cluster takes slot y.
//   Z         the merges stably sorted by height (equal heights keep merge order), then numbered as scipy does: row i joins the
//               current clusters of its two slots, (id_a < id_b, height, size), the new cluster gets id n + i.
// The caller compiles this without floating-point contraction (csrc/Makefile).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <numeric>
#include <vector>

// points[n x dim] (row-major) -> Z[(n - 1) x 4].  Returns false (Z untouched) when a distance is not finite.
inline bool linkage_complete_host(const double *points, uint32_t n, uint32_t dim, double *Z) {
    if (n < 2) return true;
    const uint64_t N = n;
    auto at = [N](uint64_t i, uint64_t j) {  // condensed index of the pair, i != j
        if (i > j) std::swap(i, j);
        return N * i - i * (i + 1) / 2 + (j - i - 1);
    };
    std::vector<double> D(N * (N - 1) / 2);
    for (uint64_t i = 0; i < N; i++)
        for (uint64_t j = i + 1; j < N; j++) {
            double s = 0.0;
            for (uint32_t c = 0; c < dim; c++) {
                const double df = points[j * dim + c] - points[i * dim + c];
                s += df * df;
            }
            const double d = std::sqrt(s);
            if (!std::isfinite(d)) return false;
            D[at(i, j)] = d;
        }
    std::vector<uint64_t> size(N, 1);
    std::vector<uint32_t> chain(N);
    std::vector<double> raw((N - 1) * 4);  // merges in merge order: slot x, slot y, height, size
    uint32_t len = 0;
    for (uint64_t k = 0; k + 1 < N; k++) {
        if (len == 0) {
            uint32_t i = 0;
            while (!size[i]) i++;
            chain[len++] = i;
        }
        uint32_t x, y = 0;
        double dmin;
        for (;;) {
            x = chain[len - 1];
            if (len > 1) {
                y = chain[len - 2];
                dmin = D[at(x, y)];
            } else {
                dmin = INFINITY;
            }
            for (uint32_t i = 0; i < n; i++) {
                if (!size[i] || i == x) continue;
                const double d = D[at(x, i)];
                if (d < dmin) {
                    dmin = d;
                    y = i;
                }
            }
            if (len > 1 && y == chain[len - 2]) break;
            chain[len++] = y;
        }
        len -= 2;
        if (x > y) std::swap(x, y);
        raw[k * 4 + 0] = x;
        raw[k * 4 + 1] = y;
        raw[k * 4 + 2] = dmin;
        raw[k * 4 + 3] = (double)(size[x] + size[y]);
        size[y] += size[x];
        size[x] = 0;
        for (uint32_t i = 0; i < n; i++) {
            if (!size[i] || i == y) continue;
            D[at(i, y)] = std::max(D[at(i, x)], D[at(i, y)]);
        }
    }
    std::vector<uint32_t> order(N - 1);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return raw[a * 4 + 2] < raw[b * 4 + 2]; });
    // union-find over slots -> cluster ids n, n + 1, ... in sorted order
    std::vector<uint64_t> parent(2 * N - 1), csize(2 * N - 1, 1);
    std::iota(parent.begin(), parent.end(), (uint64_t)0);
    auto find = [&](uint64_t v) {
        uint64_t r = v;
        while (parent[r] != r) r = parent[r];
        while (parent[v] != r) {
            const uint64_t nx = parent[v];
            parent[v] = r;
            v = nx;
        }
        return r;
    };
    for (uint64_t i = 0; i + 1 < N; i++) {
        const double *r = &raw[(uint64_t)order[i] * 4];
        const uint64_t a = find((uint64_t)r[0]), b = find((uint64_t)r[1]), id = N + i;
        parent[a] = parent[b] = id;
        csize[id] = csize[a] + csize[b];
        Z[i * 4 + 0] = (double)std::min(a, b);
        Z[i * 4 + 1] = (double)std::max(a, b);
        Z[i * 4 + 2] = r[2];
        Z[i * 4 + 3] = (double)csize[id];
    }
    return true;
}
