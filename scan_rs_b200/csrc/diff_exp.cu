// diff_exp.cu -- sSeq differential expression: the statistics of the reference's diff-exp crate (compute_sseq_params,
// sseq_differential_expression; Cell Ranger's published sSeq, which the crate ports).  The contract is restated beside the four
// entry points in include/scanb200.h and, literally, in oracle/sseq.py.
//
//   params      sb_size_factors + sb_mean_var_axis(axis 1, SizeNormalized view) of moments.cu, then O(m) host work
//   group sums  k_group_sums: one pass over the cell-major stream, u64 atomics into acc[label * m + gene]; sums_out = total - sums_in
//               (cell lists: the dual-sum kernel of moments.cu; labelled pairs: k_pair_rows picks each pair's two rows of acc)
//   exact test  the host lists the tests and cuts every sweep x = 0..T into chunks of NB_CHUNK terms; k_nb_sweep evaluates a chunk per
//               warp with online (max, sum exp) pairs over all terms and over the terms <= l_obs, k_nb_finish folds a test's chunks in
//               chunk order.  Bit-reproducible and independent of the grid: every term is a fixed function of (test, x), every chunk
//               a fixed lane / shuffle order, every fold a fixed chunk order.
//   asymptotic  k_nb_asym, a thread per test: own regularised incomplete beta (modified Lentz) and Beta median (safeguarded Newton)
//   host tail   Benjamini-Hochberg, normalized means, log2 fold changes
// Sharded contexts: every rank holds the all-reduced sums and gathers the size factors (and labels) in global cell order, so every
// rank lists the same tests with the same s_in / s_out bits; rank r evaluates a contiguous range of them (balanced by sweep chunks)
// into a zero-filled p array and one f64 all-reduce combines the ranges -- exact, each slot has one writer -- so p at any world size
// equals world 1 bit for bit given the same params.
#include <cmath>
#include <thread>

#include "common.cuh"

#define NB_CHUNK 1024              // sweep terms per warp work item
#define NB_LF_MAX ((u64)1 << 22)   // log-factorial table entries; beyond it the same lgamma is evaluated in place (bit-neutral)
#define NB_CF_MAXIT 100000         // continued-fraction cap: ~1,100 iterations at the median of Beta(1e7, 1e7), ~0.35 sqrt(alpha)

// ---------------------------------------------------------------- group sums
// warp per cell over the cell-major stream (the pattern of k_mo_int): acc[label[c] * m + gene] += count
__global__ void k_group_sums(const u64 *__restrict__ ptr, const uint2 *__restrict__ cm, u64 n, u32 m, const u32 *__restrict__ label,
                             unsigned long long *__restrict__ acc) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (u64 c = warp; c < n; c += nwarps) {
        unsigned long long *row = acc + (u64)label[c] * m;
        const u64 s = ptr[c], e = ptr[c + 1];
        for (u64 k = s + lane; k < e; k += 32) {
            const uint2 z = cm[k];
            atomicAdd(&row[z.x], (unsigned long long)z.y);
        }
    }
}

// thread per (comparison, gene): in[j] = row rows[2j] of sums, out[j] = row rows[2j + 1]
__global__ void k_pair_rows(const u64 *__restrict__ sums, u32 m, const u32 *__restrict__ rows, u32 npairs, u64 *__restrict__ in, u64 *__restrict__ out) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < (u64)npairs * m; t += (u64)gridDim.x * blockDim.x) {
        const u64 j = t / m, g = t % m;
        in[t] = sums[(u64)rows[2 * j] * m + g];
        out[t] = sums[(u64)rows[2 * j + 1] * m + g];
    }
}

// ---------------------------------------------------------------- exact test
struct NbIn {  // one exact test as the host lists it
    u64 x_in, T, slot;
    double s_in, s_out, mu, phi;
};
struct NbSide {  // the per-test constants of lp(., s): r, lgamma(r), log(mu s / (r + mu s)), r log(r / (r + mu s)); Poisson limit when phi = 0
    double r, lgr, A, B;
    int pois;
};
struct NbConst {
    NbSide in, out;
    double l_obs;
    u64 x_in, T, slot;
};

__device__ __forceinline__ double nb_lf(u64 k, const double *__restrict__ lf, u64 nlf) { return k < nlf ? lf[k] : lgamma(__dadd_rn((double)k, 1.0)); }

// lp(x, s) = lgamma(r + x) - (lgamma(r) + lgamma(x + 1)) + x A + B in this association order, no contraction
__device__ __forceinline__ double nb_lp(u64 x, const NbSide &s, const double *__restrict__ lf, u64 nlf) {
    const double xd = (double)x, f = nb_lf(x, lf, nlf);
    const double t = s.pois ? -f : __dsub_rn(lgamma(__dadd_rn(s.r, xd)), __dadd_rn(s.lgr, f));
    return __dadd_rn(__dadd_rn(t, __dmul_rn(xd, s.A)), s.B);
}
// l(x) = lp(x, s_in) + lp(T - x, s_out): the sweep term and the observed term are this one function
__device__ __forceinline__ double nb_l(u64 x, const NbConst &c, const double *__restrict__ lf, u64 nlf) {
    return __dadd_rn(nb_lp(x, c.in, lf, nlf), nb_lp(c.T - x, c.out, lf, nlf));
}

__device__ __forceinline__ NbSide nb_side(double s, double mu, double phi) {
    NbSide o;
    const double ms = __dmul_rn(s, mu);
    if (phi == 0.0) {  // Poisson limit of the NB (builder-defined): lp = -lgamma(x + 1) + x log(mu s) - mu s
        o.pois = 1;
        o.r = 0.0;
        o.lgr = 0.0;
        o.A = log(ms);
        o.B = -ms;
    } else {
        o.pois = 0;
        o.r = __ddiv_rn(s, phi);
        o.lgr = lgamma(o.r);
        const double rm = __dadd_rn(o.r, ms);
        o.A = log(__ddiv_rn(ms, rm));
        o.B = __dmul_rn(o.r, log(__ddiv_rn(o.r, rm)));
    }
    return o;
}

__global__ void k_lf_table(double *__restrict__ lf, u64 n) {
    for (u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (u64)gridDim.x * blockDim.x) lf[k] = lgamma(__dadd_rn((double)k, 1.0));
}

__global__ void k_nb_prep(const NbIn *__restrict__ in, u64 nt, const double *__restrict__ lf, u64 nlf, NbConst *__restrict__ out) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += (u64)gridDim.x * blockDim.x) {
        const NbIn a = in[t];
        NbConst c;
        c.in = nb_side(a.s_in, a.mu, a.phi);
        c.out = nb_side(a.s_out, a.mu, a.phi);
        c.x_in = a.x_in;
        c.T = a.T;
        c.slot = a.slot;
        c.l_obs = nb_l(a.x_in, c, lf, nlf);
        out[t] = c;
    }
}

// chunk -> test map from the per-test first chunk
__global__ void k_chunk_map(const u64 *__restrict__ chunk0, u64 nt, u32 *__restrict__ chunk_test) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += (u64)gridDim.x * blockDim.x)
        for (u64 k = chunk0[t]; k < chunk0[t + 1]; k++) chunk_test[k] = (u32)t;
}

// online log-sum-exp: (m, s) represents m + log(s); s == 0 is the empty set
__device__ __forceinline__ void lse_push(double &m, double &s, double l) {
    if (l > m) {
        s = s * exp(m - l) + 1.0;
        m = l;
    } else {
        s += exp(l - m);
    }
}
__device__ __forceinline__ void lse_merge(double &m, double &s, double m2, double s2) {
    if (s2 == 0.0) return;
    if (s == 0.0) {
        m = m2;
        s = s2;
    } else if (m2 > m) {
        s = s * exp(m - m2) + s2;
        m = m2;
    } else {
        s += s2 * exp(m2 - m);
    }
}

// a warp per chunk of NB_CHUNK terms: lane l takes x0 + l, x0 + l + 32, ...; out[chunk] = (max, sum) over all terms, (max, sum) over l <= l_obs
__global__ void __launch_bounds__(256) k_nb_sweep(const NbConst *__restrict__ tc, const u64 *__restrict__ chunk0, const u32 *__restrict__ chunk_test,
                                                  u64 nchunks, const double *__restrict__ lf, u64 nlf, double4 *__restrict__ out) {
    u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u64 nwarps = ((u64)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (u64 ch = warp; ch < nchunks; ch += nwarps) {
        const u32 t = chunk_test[ch];
        const NbConst c = tc[t];
        const u64 x0 = (ch - chunk0[t]) * NB_CHUNK, x1 = min(x0 + NB_CHUNK, c.T + 1);
        double ma = -INFINITY, sa = 0.0, ml = -INFINITY, sl = 0.0;
        for (u64 x = x0 + lane; x < x1; x += 32) {
            const double l = nb_l(x, c, lf, nlf);
            lse_push(ma, sa, l);
            if (l <= c.l_obs) lse_push(ml, sl, l);
        }
        for (int o = 16; o > 0; o >>= 1) {
            const double ma2 = __shfl_xor_sync(0xffffffffu, ma, o), sa2 = __shfl_xor_sync(0xffffffffu, sa, o);
            const double ml2 = __shfl_xor_sync(0xffffffffu, ml, o), sl2 = __shfl_xor_sync(0xffffffffu, sl, o);
            lse_merge(ma, sa, ma2, sa2);
            lse_merge(ml, sl, ml2, sl2);
        }
        if (lane == 0) out[ch] = make_double4(ma, sa, ml, sl);
    }
}

// a thread per test: fold its chunks in chunk order, p = exp(LSE_le - LSE_all) into p[slot]
__global__ void k_nb_finish(const NbConst *__restrict__ tc, const u64 *__restrict__ chunk0, u64 nt, const double4 *__restrict__ part, double *__restrict__ p) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += (u64)gridDim.x * blockDim.x) {
        double ma = -INFINITY, sa = 0.0, ml = -INFINITY, sl = 0.0;
        for (u64 k = chunk0[t]; k < chunk0[t + 1]; k++) {
            const double4 v = part[k];
            lse_merge(ma, sa, v.x, v.y);
            lse_merge(ml, sl, v.z, v.w);
        }
        p[tc[t].slot] = sl > 0.0 ? exp((ml + log(sl)) - (ma + log(sa))) : 0.0;
    }
}

// ---------------------------------------------------------------- asymptotic test
// continued fraction of I_x(a, b) (modified Lentz; Numerical Recipes 6.4 betacf)
__device__ double beta_cf(double a, double b, double x, int *bad) {
    const double FPMIN = 1e-300, EPS = 1e-15;
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    double c = 1.0, d = 1.0 - qab * x / qap;
    if (fabs(d) < FPMIN) d = FPMIN;
    d = 1.0 / d;
    double h = d;
    for (int it = 1; it <= NB_CF_MAXIT; it++) {
        const double mm = (double)it, m2 = 2.0 * mm;
        double aa = mm * (b - mm) * x / ((qam + m2) * (a + m2));
        d = 1.0 + aa * d;
        if (fabs(d) < FPMIN) d = FPMIN;
        c = 1.0 + aa / c;
        if (fabs(c) < FPMIN) c = FPMIN;
        d = 1.0 / d;
        h *= d * c;
        aa = -(a + mm) * (qab + mm) * x / ((a + m2) * (qap + m2));
        d = 1.0 + aa * d;
        if (fabs(d) < FPMIN) d = FPMIN;
        c = 1.0 + aa / c;
        if (fabs(c) < FPMIN) c = FPMIN;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < EPS) return h;
    }
    *bad = 1;
    return h;
}
// I_x(a, b) and its complement 1 - I_x(a, b) = I_{1-x}(b, a), each from the side of the symmetry switch x = (a + 1) / (a + b + 2)
// where the fraction converges; prefactor x^a (1 - x)^b / B(a, b) through lgamma
__device__ void beta_inc(double a, double b, double x, double lbeta, double &I, double &Ic, int *bad) {
    if (x <= 0.0) {
        I = 0.0;
        Ic = 1.0;
        return;
    }
    if (x >= 1.0) {
        I = 1.0;
        Ic = 0.0;
        return;
    }
    const double bt = exp(a * log(x) + b * log1p(-x) - lbeta);
    if (x < (a + 1.0) / (a + b + 2.0)) {
        I = bt * beta_cf(a, b, x, bad) / a;
        Ic = 1.0 - I;
    } else {
        Ic = bt * beta_cf(b, a, 1.0 - x, bad) / b;
        I = 1.0 - Ic;
    }
}
// median of Beta(a, b): Newton on I_x(a, b) = 1/2 from (a - 1/3) / (a + b - 2/3), kept inside the bracket by bisection
__device__ double beta_median(double a, double b, double lbeta, int *bad) {
    double lo = 0.0, hi = 1.0, x = (a - 1.0 / 3.0) / (a + b - 2.0 / 3.0);
    if (!(x > 0.0 && x < 1.0)) x = a / (a + b);
    for (int it = 0; it < 400; it++) {
        double I, Ic;
        beta_inc(a, b, x, lbeta, I, Ic, bad);
        const double f = I < 0.5 ? I - 0.5 : 0.5 - Ic;
        if (f == 0.0) return x;
        if (f < 0.0) lo = x;
        else hi = x;
        const double pdf = exp((a - 1.0) * log(x) + (b - 1.0) * log1p(-x) - lbeta);
        double xn = x - f / pdf;
        if (!(xn > lo && xn < hi)) xn = 0.5 * (lo + hi);
        if (fabs(xn - x) <= 1e-15 * x || hi - lo <= 1e-15 * x) return xn;
        x = xn;
    }
    *bad = 1;
    return x;
}

__global__ void k_nb_asym(const NbIn *__restrict__ in, u64 nt, double *__restrict__ p, int *__restrict__ bad_flag) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += (u64)gridDim.x * blockDim.x) {
        const NbIn q = in[t];
        int bad = 0;
        const double x_in = (double)q.x_in, T = x_in + (double)(q.T - q.x_in);
        const double alpha = q.s_in * q.mu / (1.0 + q.phi * q.mu);
        const double beta = (q.s_out / q.s_in) * alpha;
        const double lbeta = lgamma(alpha) + lgamma(beta) - lgamma(alpha + beta);
        const double med = beta_median(alpha, beta, lbeta, &bad);
        const double xl = (x_in + 0.5) / T;
        double I, Ic, r;
        if (xl < med) {
            beta_inc(alpha, beta, xl, lbeta, I, Ic, &bad);
            r = 2.0 * I;
        } else {
            beta_inc(alpha, beta, (x_in - 0.5) / T, lbeta, I, Ic, &bad);
            r = 2.0 * Ic;
        }
        p[q.slot] = r;
        if (bad) atomicOr(bad_flag, 1);
    }
}

// ---------------------------------------------------------------- host side
static int de_grid(sb_ctx *ctx, u64 items, int per_block) {
    return (int)std::max<u64>(1, std::min<u64>((items + per_block - 1) / per_block, (u64)ctx->sm_count * 16));
}

int group_gene_sums(sb_mat *mat, const u32 *d_lab, u32 n_groups, DevBuf<u64> &acc) {
    sb_ctx *ctx = mat->ctx;
    const u64 cells = (u64)n_groups * mat->m;
    SB_TRY(acc.alloc(cells));
    SB_CUDA(cudaMemsetAsync(acc.p, 0, cells * sizeof(u64), ctx->stream));
    if (mat->n && mat->nnz) {
        ProfScope ps(ctx, PH_REDUCE);
        k_group_sums<<<de_grid(ctx, mat->n * 32, 256), 256, 0, ctx->stream>>>(mat->cm_ptr.p, mat->cm.p, mat->n, mat->m, d_lab, (unsigned long long *)acc.p);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
    }
    return comm_allreduce_u64(ctx, acc.p, cells);
}

// one value per local cell -> the values of all cells in global cell order (zero-padded f64 all-reduce: one writer per slot, exact)
int gather_cells(sb_ctx *ctx, const std::vector<double> &mine, std::vector<double> &all) {
    if (ctx->nranks == 1) {
        all = mine;
        return SB_OK;
    }
    std::vector<u64> counts;
    SB_TRY(comm_allgather_u64_host(ctx, mine.size(), counts));
    u64 total = 0, off = 0;
    for (int r = 0; r < ctx->nranks; r++) {
        if (r < ctx->rank) off += counts[r];
        total += counts[r];
    }
    all.assign(total, 0.0);
    std::copy(mine.begin(), mine.end(), all.begin() + off);
    DevBuf<double> d;
    SB_TRY(d.alloc(std::max<u64>(1, total)));
    if (total) SB_CUDA(cudaMemcpyAsync(d.p, all.data(), total * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    SB_TRY(comm_allreduce_f64(ctx, d.p, total));
    if (total) SB_CUDA(cudaMemcpyAsync(all.data(), d.p, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    return SB_OK;
}

int sseq_check_params(sb_mat *mat, const sb_sseq_params *p, const char *fn) {
    if (!p || !p->size_factors || !p->gene_means || !p->gene_phi || !p->use_genes) return sb_fail(SB_ERR_INVALID_ARG, "%s: NULL params array", fn);
    if (p->num_genes != mat->m || p->num_cells != mat->n_global)
        return sb_fail(SB_ERR_INVALID_ARG, "%s: params are for %u genes x %llu cells, the matrix has %u x %llu", fn, p->num_genes,
                       (unsigned long long)p->num_cells, mat->m, (unsigned long long)mat->n_global);
    return SB_OK;
}

// Benjamini-Hochberg (Cell Ranger's adjust_pvalue_bh): q = min(1, cummin over descending p of p n / rank); tied p share one q
static void bh_adjust(const double *p, u64 n, double *q) {
    std::vector<u64> order(n);
    for (u64 i = 0; i < n; i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](u64 a, u64 b) { return p[a] > p[b]; });
    double run = INFINITY;
    for (u64 i = 0; i < n; i++) {
        const u64 k = n - i;  // rank in ascending order
        const double v = (double)n / (double)k * p[order[i]];
        run = std::min(run, v);
        q[order[i]] = std::min(1.0, run);
    }
}

// The test stage shared by both entries: sums [ncomp x m] (replicated), s_in / s_out per comparison -> every output array.
static int sseq_tests(sb_mat *mat, const sb_sseq_params *prm, u32 ncomp, const std::vector<double> &s_in, const std::vector<double> &s_out,
                      u64 big_count, sb_diff_exp_out *out) {
    sb_ctx *ctx = mat->ctx;
    const u32 m = mat->m;
    const u64 total = (u64)ncomp * m;
    // list the tests (identical on every rank)
    TraceScope tr_stage(ctx, "sseq: test stage");
    std::vector<NbIn> ex, as;
    std::vector<u64> ex_chunks;
    ex.reserve(total);
    ex_chunks.reserve(total);
    for (u32 j = 0; j < ncomp; j++)
        for (u32 g = 0; g < m; g++) {
            if (!prm->use_genes[g]) continue;
            const u64 slot = (u64)j * m + g, xi = out->sums_in[slot], xo = out->sums_out[slot];
            const NbIn t{xi, xi + xo, slot, s_in[j], s_out[j], prm->gene_means[g], prm->gene_phi[g]};
            if (xi > big_count && xo > big_count) {
                as.push_back(t);
            } else {
                ex.push_back(t);
                ex_chunks.push_back((xi + xo) / NB_CHUNK + 1);
            }
        }
    // this rank's contiguous ranges: exact tests balanced by sweep chunks, asymptotic tests by count
    const int R = ctx->nranks, rk = ctx->rank;
    u64 all_chunks = 0;
    for (u64 c : ex_chunks) all_chunks += c;
    u64 e_lo = 0, e_hi = ex.size();
    if (R > 1) {
        const u64 want_lo = all_chunks * (u64)rk / R, want_hi = all_chunks * (u64)(rk + 1) / R;
        u64 acc = 0;
        e_lo = e_hi = ex.size();
        bool have_lo = false;
        for (u64 t = 0; t < ex.size(); t++) {
            if (!have_lo && acc >= want_lo) {
                e_lo = t;
                have_lo = true;
            }
            if (acc >= want_hi) {
                e_hi = t;
                break;
            }
            acc += ex_chunks[t];
        }
        if (!have_lo) e_lo = ex.size();
        if (rk == R - 1) e_hi = ex.size();
        if (e_hi < e_lo) e_hi = e_lo;
    }
    const u64 a_lo = as.size() * (u64)rk / R, a_hi = as.size() * (u64)(rk + 1) / R;
    const u64 ne = e_hi - e_lo, na = a_hi - a_lo;

    DevBuf<double> p;
    SB_TRY(p.alloc(std::max<u64>(1, total)));
    SB_CUDA(cudaMemsetAsync(p.p, 0, std::max<u64>(1, total) * sizeof(double), ctx->stream));
    DevBuf<int> bad;
    SB_TRY(bad.alloc(1));
    SB_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), ctx->stream));
    if (ne) {
        TraceScope tr(ctx, "sseq: exact sweep");
        std::vector<u64> chunk0(ne + 1, 0);
        u64 maxT = 0;
        for (u64 i = 0; i < ne; i++) {
            chunk0[i + 1] = chunk0[i] + ex_chunks[e_lo + i];
            maxT = std::max(maxT, ex[e_lo + i].T);
        }
        const u64 nch = chunk0[ne], nlf = std::min<u64>(maxT + 1, NB_LF_MAX);
        DevBuf<NbIn> d_in;
        DevBuf<NbConst> d_c;
        DevBuf<u64> d_c0;
        DevBuf<u32> d_map;
        DevBuf<double> d_lf;
        DevBuf<double4> d_part;
        SB_TRY(d_in.alloc(ne));
        SB_TRY(d_c.alloc(ne));
        SB_TRY(d_c0.alloc(ne + 1));
        SB_TRY(d_map.alloc(nch));
        SB_TRY(d_lf.alloc(nlf));
        SB_TRY(d_part.alloc(nch));
        SB_CUDA(cudaMemcpyAsync(d_in.p, ex.data() + e_lo, ne * sizeof(NbIn), cudaMemcpyHostToDevice, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(d_c0.p, chunk0.data(), (ne + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        k_lf_table<<<de_grid(ctx, nlf, 256), 256, 0, ctx->stream>>>(d_lf.p, nlf);
        k_nb_prep<<<de_grid(ctx, ne, 128), 128, 0, ctx->stream>>>(d_in.p, ne, d_lf.p, nlf, d_c.p);
        k_chunk_map<<<de_grid(ctx, ne, 256), 256, 0, ctx->stream>>>(d_c0.p, ne, d_map.p);
        k_nb_sweep<<<de_grid(ctx, nch, 8), 256, 0, ctx->stream>>>(d_c.p, d_c0.p, d_map.p, nch, d_lf.p, nlf, d_part.p);
        k_nb_finish<<<de_grid(ctx, ne, 128), 128, 0, ctx->stream>>>(d_c.p, d_c0.p, ne, d_part.p, p.p);
        for (int i = 0; i < 5; i++) count_launch(ctx);
        SB_CUDA(cudaGetLastError());
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    if (na) {
        TraceScope tr(ctx, "sseq: asymptotic");
        DevBuf<NbIn> d_in;
        SB_TRY(d_in.alloc(na));
        SB_CUDA(cudaMemcpyAsync(d_in.p, as.data() + a_lo, na * sizeof(NbIn), cudaMemcpyHostToDevice, ctx->stream));
        k_nb_asym<<<de_grid(ctx, na, 128), 128, 0, ctx->stream>>>(d_in.p, na, p.p, bad.p);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    TraceScope tr(ctx, "sseq: p all-reduce + host tail");
    SB_TRY(comm_allreduce_f64(ctx, p.p, total));
    int hbad = 0;
    SB_CUDA(cudaMemcpyAsync(out->p_values, p.p, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaMemcpyAsync(&hbad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
    SB_TRY(agree_status(ctx, hbad ? sb_fail(SB_ERR_LINALG, "sSeq asymptotic test: the incomplete beta function did not converge") : SB_OK, "sSeq test"));
    // host tail, one comparison per host thread at a time (each writes its own rows)
    auto tail = [&](u32 j) {
        std::vector<double> pt;
        std::vector<u64> idx;
        const u64 o = (u64)j * m;
        for (u32 g = 0; g < m; g++) {
            const u64 i = o + g;
            const double xi = (double)out->sums_in[i], xo = (double)out->sums_out[i];
            out->normalized_mean_in[i] = xi / s_in[j];
            out->normalized_mean_out[i] = xo / s_out[j];
            out->log2_fold_change[i] = std::log2((1.0 + xi) / (1.0 + s_in[j])) - std::log2((1.0 + xo) / (1.0 + s_out[j]));
            if (!prm->use_genes[g]) out->p_values[i] = 1.0;
            out->adjusted_p_values[i] = out->p_values[i];
            if (prm->use_genes[g]) {
                pt.push_back(out->p_values[i]);
                idx.push_back(i);
            }
        }
        std::vector<double> q(pt.size());
        bh_adjust(pt.data(), pt.size(), q.data());
        for (size_t k = 0; k < idx.size(); k++) out->adjusted_p_values[idx[k]] = q[k];
    };
    const u32 nth = std::min<u32>(ncomp, std::max(1u, std::min(16u, std::thread::hardware_concurrency())));
    if (nth <= 1) {
        for (u32 j = 0; j < ncomp; j++) tail(j);
    } else {
        std::vector<std::thread> th;
        for (u32 t = 0; t < nth; t++)
            th.emplace_back([&, t] {
                for (u32 j = t; j < ncomp; j += nth) tail(j);
            });
        for (auto &x : th) x.join();
    }
    return SB_OK;
}

int sseq_pair_tests(sb_mat *mat, const sb_sseq_params *prm, const u64 *d_sums, const std::vector<u32> &rows, const std::vector<double> &s_in,
                    const std::vector<double> &s_out, u64 big_count, sb_diff_exp_out *out) {
    sb_ctx *ctx = mat->ctx;
    const u32 m = mat->m, np = (u32)s_in.size();
    const u64 total = (u64)np * m;
    {
        DevBuf<u32> d_rows;
        DevBuf<u64> d_in, d_out;
        SB_TRY(d_rows.alloc(2 * (u64)np));
        SB_TRY(d_in.alloc(total));
        SB_TRY(d_out.alloc(total));
        SB_CUDA(cudaMemcpyAsync(d_rows.p, rows.data(), 2 * (u64)np * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        k_pair_rows<<<de_grid(ctx, total, 256), 256, 0, ctx->stream>>>(d_sums, m, d_rows.p, np, d_in.p, d_out.p);
        count_launch(ctx);
        SB_CUDA(cudaGetLastError());
        SB_CUDA(cudaMemcpyAsync(out->sums_in, d_in.p, total * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaMemcpyAsync(out->sums_out, d_out.p, total * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return sseq_tests(mat, prm, np, s_in, s_out, big_count, out);
}

static bool de_out_ok(const sb_diff_exp_out *o) {
    return o && o->sums_in && o->sums_out && o->normalized_mean_in && o->normalized_mean_out && o->p_values && o->adjusted_p_values && o->log2_fold_change;
}

extern "C" int sb_sseq_compute_params(sb_mat *mat, double zeta_quantile, sb_sseq_params *out) {
    if (!mat || !out || !out->size_factors || !out->gene_means || !out->gene_variances || !out->gene_moment_phi || !out->gene_phi || !out->use_genes ||
        !(zeta_quantile >= 0.0 && zeta_quantile <= 1.0))
        return sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_compute_params: bad argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    const u32 m = mat->m;
    double *sf = out->size_factors;
    SB_TRY(sb_size_factors(mat, nullptr, 0, nullptr, sf));
    int rc = SB_OK;
    for (u64 c = 0; c < mat->n; c++)
        if (!(sf[c] > 0.0)) {
            rc = sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_compute_params: cell %llu has a total of 0 (its size factor is 0 and sum 1/sf is infinite)",
                         (unsigned long long)(mat->cell_offset + c));
            break;
        }
    SB_TRY(agree_status(ctx, rc, "sb_sseq_compute_params"));
    SB_TRY(sb_mean_var_axis(mat, 1, sf, out->gene_means, out->gene_variances));
    std::vector<double> all;
    SB_TRY(gather_cells(ctx, std::vector<double>(sf, sf + mat->n), all));
    double S = 0.0;
    for (double v : all) S += 1.0 / v;  // global cell order: the same bits at every rank count
    const double N = (double)mat->n_global, G = (double)m;
    std::vector<double> used;
    for (u32 g = 0; g < m; g++) {
        const double mu = out->gene_means[g], var = out->gene_variances[g];
        out->use_genes[g] = var > 0.0;
        out->gene_moment_phi[g] = 0.0;
        if (var > 0.0) {
            out->gene_moment_phi[g] = std::max(0.0, (N * var - mu * S) / ((mu * mu) * S));
            used.push_back(out->gene_moment_phi[g]);
        }
    }
    if (used.empty()) return sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_compute_params: no gene has a non-zero variance");
    double mean_phi = 0.0, any_pos = 0.0;
    for (double v : used) {
        mean_phi += v;
        any_pos += v > 0.0;
    }
    mean_phi /= (double)used.size();
    std::vector<double> sorted = used;
    const double zeta = percentile_of(sorted, zeta_quantile);
    double num = 0.0, den = 0.0;
    for (double v : used) {
        num += (v - mean_phi) * (v - mean_phi);
        den += (v - zeta) * (v - zeta);
    }
    const double delta = (num / (G - 1.0)) / (den / (G - 2.0));
    for (u32 g = 0; g < m; g++) {
        if (!out->use_genes[g]) out->gene_phi[g] = NAN;
        else out->gene_phi[g] = any_pos > 0.0 ? (1.0 - delta) * out->gene_moment_phi[g] + delta * zeta : 0.0;
    }
    out->num_cells = mat->n_global;
    out->num_genes = m;
    out->reserved = 0;
    out->zeta_hat = zeta;
    out->delta = delta;
    return SB_OK;
}

extern "C" int sb_sseq_diff_exp(sb_mat *mat, const sb_sseq_params *params, const uint64_t *cond_in, uint64_t n_in, const uint64_t *cond_out,
                                uint64_t n_out, uint64_t big_count, sb_diff_exp_out *out) {
    if (!mat || !de_out_ok(out) || (!cond_in && n_in) || (!cond_out && n_out)) return sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_diff_exp: bad argument");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    int rc = sseq_check_params(mat, params, "sb_sseq_diff_exp");
    const uint64_t *lists[2] = {cond_in, cond_out};
    const uint64_t lens[2] = {n_in, n_out};
    for (int l = 0; l < 2 && rc == SB_OK; l++)
        for (u64 i = 0; i < lens[l]; i++) {
            if (lists[l][i] >= mat->n) {
                rc = sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_diff_exp: cell index %llu out of range (%llu local cells)", (unsigned long long)lists[l][i],
                             (unsigned long long)mat->n);
                break;
            }
            if (i && lists[l][i] <= lists[l][i - 1]) {
                rc = sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_diff_exp: cell list %s is not strictly ascending at position %llu", l ? "cond_out" : "cond_in",
                             (unsigned long long)i);
                break;
            }
        }
    SB_TRY(agree_status(ctx, rc, "sb_sseq_diff_exp"));
    // s_in / s_out: the listed cells' size factors summed in global cell order (unlisted cells contribute an exact +0)
    std::vector<double> w_in(mat->n, 0.0), w_out(mat->n, 0.0), all_in, all_out;
    for (u64 i = 0; i < n_in; i++) w_in[cond_in[i]] = params->size_factors[cond_in[i]];
    for (u64 i = 0; i < n_out; i++) w_out[cond_out[i]] = params->size_factors[cond_out[i]];
    SB_TRY(gather_cells(ctx, w_in, all_in));
    SB_TRY(gather_cells(ctx, w_out, all_out));
    std::vector<u64> len_in, len_out;  // list lengths of every rank
    SB_TRY(comm_allgather_u64_host(ctx, n_in, len_in));
    SB_TRY(comm_allgather_u64_host(ctx, n_out, len_out));
    u64 cnt_in = 0, cnt_out = 0;
    for (u64 v : len_in) cnt_in += v;
    for (u64 v : len_out) cnt_out += v;
    if (!cnt_in || !cnt_out) return sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_diff_exp: condition %s is empty", cnt_in ? "cond_out" : "cond_in");
    std::vector<double> s_in(1, 0.0), s_out(1, 0.0);
    for (double v : all_in) s_in[0] += v;
    for (double v : all_out) s_out[0] += v;
    {
        TraceScope tr(ctx, "sseq: group sums");
        SB_TRY(sb_sum_rows_dual(mat, cond_in, n_in, cond_out, n_out, out->sums_in, out->sums_out));
    }
    return sseq_tests(mat, params, 1, s_in, s_out, big_count, out);
}

extern "C" int sb_sseq_one_vs_rest(sb_mat *mat, const sb_sseq_params *params, const uint32_t *labels, uint32_t n_groups, uint64_t big_count,
                                   sb_diff_exp_out *out) {
    if (!mat || !de_out_ok(out) || (!labels && mat->n) || n_groups < 2) return sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_one_vs_rest: bad argument (n_groups >= 2)");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    const u32 m = mat->m;
    int rc = sseq_check_params(mat, params, "sb_sseq_one_vs_rest");
    for (u64 c = 0; c < mat->n && rc == SB_OK; c++)
        if (labels[c] >= n_groups)
            rc = sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_one_vs_rest: label %u of cell %llu is not below n_groups = %u", labels[c],
                         (unsigned long long)(mat->cell_offset + c), n_groups);
    SB_TRY(agree_status(ctx, rc, "sb_sseq_one_vs_rest"));
    // labels and size factors of all cells in global cell order: group sizes and s_in / s_out, the same bits on every rank
    std::vector<u64> size(n_groups, 0);
    std::vector<double> s_in(n_groups, 0.0), s_out(n_groups, 0.0);
    {
        TraceScope tr(ctx, "sseq: cell gathers");
        std::vector<double> lab_l(mat->n), lab, sf;
        for (u64 c = 0; c < mat->n; c++) lab_l[c] = (double)labels[c];
        SB_TRY(gather_cells(ctx, lab_l, lab));
        SB_TRY(gather_cells(ctx, std::vector<double>(params->size_factors, params->size_factors + mat->n), sf));
        // every accumulator adds in global cell order; a cell outside a comparison's rest group adds an exact +0
        for (u64 c = 0; c < lab.size(); c++) {
            const u32 l = (u32)lab[c];
            const double v = sf[c];
            size[l]++;
            s_in[l] += v;
            for (u32 j = 0; j < n_groups; j++) s_out[j] += j == l ? 0.0 : v;
        }
    }
    for (u32 j = 0; j < n_groups; j++)
        if (!size[j]) return sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_one_vs_rest: group %u is empty", j);
    {
        TraceScope tr(ctx, "sseq: group sums");
        const u64 cells = (u64)n_groups * m;
        DevBuf<u32> d_lab;
        DevBuf<u64> acc;
        SB_TRY(d_lab.alloc(std::max<u64>(1, mat->n)));
        if (mat->n) SB_CUDA(cudaMemcpyAsync(d_lab.p, labels, mat->n * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        SB_TRY(group_gene_sums(mat, d_lab.p, n_groups, acc));
        SB_CUDA(cudaMemcpyAsync(out->sums_in, acc.p, cells * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        SB_CUDA(cudaStreamSynchronize(ctx->stream));
        std::vector<u64> tot(m, 0);
        for (u32 j = 0; j < n_groups; j++)
            for (u32 g = 0; g < m; g++) tot[g] += out->sums_in[(u64)j * m + g];
        for (u32 j = 0; j < n_groups; j++)
            for (u32 g = 0; g < m; g++) out->sums_out[(u64)j * m + g] = tot[g] - out->sums_in[(u64)j * m + g];
    }
    return sseq_tests(mat, params, n_groups, s_in, s_out, big_count, out);
}

extern "C" int sb_sseq_pairs(sb_mat *mat, const sb_sseq_params *params, const uint32_t *labels, uint32_t n_groups, const uint32_t *pairs,
                             uint32_t n_pairs, uint64_t big_count, sb_diff_exp_out *out) {
    if (!mat || !de_out_ok(out) || (!labels && mat->n) || !pairs || !n_pairs) return sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_pairs: bad argument (n_pairs >= 1)");
    sb_ctx *ctx = mat->ctx;
    SB_ENTER(ctx);
    int rc = sseq_check_params(mat, params, "sb_sseq_pairs");
    for (u32 j = 0; j < n_pairs && rc == SB_OK; j++)
        if (pairs[2 * j] == pairs[2 * j + 1] || pairs[2 * j] >= n_groups || pairs[2 * j + 1] >= n_groups)
            rc = sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_pairs: pair %u = (%u, %u) needs two different groups below n_groups = %u", j, pairs[2 * j],
                         pairs[2 * j + 1], n_groups);
    for (u64 c = 0; c < mat->n && rc == SB_OK; c++)
        if (labels[c] >= n_groups)
            rc = sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_pairs: label %u of cell %llu is not below n_groups = %u", labels[c],
                         (unsigned long long)(mat->cell_offset + c), n_groups);
    SB_TRY(agree_status(ctx, rc, "sb_sseq_pairs"));
    // s of every group: its size factors summed in global cell order (the bits sb_sseq_diff_exp gets with the group's cell list)
    std::vector<u64> size(n_groups, 0);
    std::vector<double> s(n_groups, 0.0);
    {
        TraceScope tr(ctx, "sseq: cell gathers");
        std::vector<double> lab_l(mat->n), lab, sf;
        for (u64 c = 0; c < mat->n; c++) lab_l[c] = (double)labels[c];
        SB_TRY(gather_cells(ctx, lab_l, lab));
        SB_TRY(gather_cells(ctx, std::vector<double>(params->size_factors, params->size_factors + mat->n), sf));
        for (u64 c = 0; c < lab.size(); c++) {
            size[(u32)lab[c]]++;
            s[(u32)lab[c]] += sf[c];
        }
    }
    std::vector<double> s_in(n_pairs), s_out(n_pairs);
    std::vector<u32> rows(pairs, pairs + 2 * (u64)n_pairs);
    for (u32 j = 0; j < n_pairs; j++) {
        for (int h = 0; h < 2; h++)
            if (!size[pairs[2 * j + h]]) return sb_fail(SB_ERR_INVALID_ARG, "sb_sseq_pairs: group %u (pair %u) is empty", pairs[2 * j + h], j);
        s_in[j] = s[pairs[2 * j]];
        s_out[j] = s[pairs[2 * j + 1]];
    }
    DevBuf<u64> acc;
    {
        TraceScope tr(ctx, "sseq: group sums");
        DevBuf<u32> d_lab;
        SB_TRY(d_lab.alloc(std::max<u64>(1, mat->n)));
        if (mat->n) SB_CUDA(cudaMemcpyAsync(d_lab.p, labels, mat->n * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
        SB_TRY(group_gene_sums(mat, d_lab.p, n_groups, acc));
    }
    return sseq_pair_tests(mat, params, acc.p, rows, s_in, s_out, big_count, out);
}
