// scanb200.hpp -- header-only C++ host layer over the C ABI (scanb200.h).
//
// The reference is a Rust workspace and no Rust toolchain exists in this image, so the host side
// above the C ABI is written in C++ and mirrors the reference's interface for this path: same
// module layout as namespaces (sqz, normalization, dim_red, snoop), same type and function names,
// same argument meaning, same error messages.  A Rust crate would wrap the same C symbols the same
// way (INTEGRATION.md).  Everything here is thin: all logic lives behind the C ABI.
//
//   reference                                                    here
//   sqz::AdaptiveMat<u32>            sqz/src/mat.rs:34-42         scanb200::sqz::AdaptiveMat
//   sqz::LowRankOffset               sqz/src/low_rank_offset.rs   scanb200::sqz::LowRankOffset
//   scan_rs::normalization::*        scan-rs/src/normalization.rs scanb200::normalization::*
//   scan_rs::dim_red::{Pca,BkSvd,..} scan-rs/src/dim_red/*.rs     scanb200::dim_red::*
//   snoop::{CancelProgress,NoOpSnoop} snoop/src/lib.rs            scanb200::snoop::*
//   diff_exp::{compute_sseq_params,..} diff-exp/src/diff_exp.rs   scanb200::diff_exp::*
//   leiden (Louvain), SNN graph      leiden crate (deterministic)  scanb200::clustering::*
//   umap-rs (UMAP)                   umap-rs crate (deterministic) scanb200::embedding::*
//   bhtsne (t-SNE)                   bhtsne crate (deterministic)  scanb200::embedding::tsne*
#pragma once
#include <type_traits>
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "scanb200.h"

namespace scanb200 {

// anyhow::Error carrying the library message; CancellationError mirrors snoop::CancellationError
struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &msg) : std::runtime_error(msg), code(c) {}
};
struct CancellationError : Error {
    using Error::Error;
};

inline void check(int rc) {
    if (rc == SB_OK) return;
    std::string msg = sb_last_error();
    if (rc == SB_ERR_CANCELLED) throw CancellationError(rc, msg);
    throw Error(rc, msg);
}

// ndarray::Array2<f64> in standard (row-major) layout
struct Array2 {
    size_t rows = 0, cols = 0;
    std::vector<double> data;
    Array2() {}
    Array2(size_t r, size_t c) : rows(r), cols(c), data(r * c, 0.0) {}
    double &operator()(size_t r, size_t c) { return data[r * cols + c]; }
    double operator()(size_t r, size_t c) const { return data[r * cols + c]; }
    std::array<size_t, 2> shape() const { return {rows, cols}; }
};

class Context {
  public:
    explicit Context(int device = 0) { check(sb_init(device, &h_)); }
    ~Context() {
        if (h_) sb_shutdown(h_);
    }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    static std::array<char, 128> unique_id() {
        std::array<char, 128> id{};
        check(sb_comm_unique_id(id.data()));
        return id;
    }
    void comm_init(int nranks, int rank, const std::array<char, 128> &id) { check(sb_comm_init(h_, nranks, rank, id.data())); }
    void set_option(const char *name, double v) { check(sb_set_option(h_, name, v)); }
    sb_ctx *raw() const { return h_; }

  private:
    sb_ctx *h_ = nullptr;
};

namespace snoop {
// snoop::CancelProgress (snoop/src/lib.rs:37-58): is_cancelled + set_progress; set_progress_check is
// implemented once in the callback trampoline below.
struct CancelProgress {
    virtual ~CancelProgress() {}
    virtual bool is_cancelled() const = 0;
    virtual void set_progress(double fraction) = 0;
};
struct NoOpSnoop : CancelProgress {  // snoop/src/lib.rs:60-85
    bool is_cancelled() const override { return false; }
    void set_progress(double) override {}
};
inline int trampoline(double fraction, void *user) {
    auto *s = static_cast<CancelProgress *>(user);
    if (s->is_cancelled()) return 1;  // Err(CancellationError) before the progress is recorded (:50-56)
    s->set_progress(fraction);
    return 0;
}
}  // namespace snoop

namespace sqz {

class LowRankOffset;

// AdaptiveMat<u32>: the count matrix, features (rows) x barcodes (cols), resident on the device.
class AdaptiveMat {
  public:
    using Partition = std::tuple<AdaptiveMat, AdaptiveMat, std::vector<size_t>, std::vector<size_t>>;

    // from_csmat on CSR arrays: indptr over genes (sqz/src/mat.rs:92-124)
    static AdaptiveMat from_csr(Context &ctx, uint32_t rows, uint64_t cols, const std::vector<uint64_t> &indptr, const std::vector<uint32_t> &idx,
                                const std::vector<uint32_t> &val) {
        sb_mat *h = nullptr;
        check(sb_upload(ctx.raw(), SB_GENE_MAJOR, rows, cols, indptr.data(), idx.data(), val.data(), &h));
        return AdaptiveMat(h);
    }
    // CSC arrays: indptr over cells
    static AdaptiveMat from_csc(Context &ctx, uint32_t rows, uint64_t cols, const std::vector<uint64_t> &indptr, const std::vector<uint32_t> &idx,
                                const std::vector<uint32_t> &val) {
        sb_mat *h = nullptr;
        check(sb_upload(ctx.raw(), SB_CELL_MAJOR, rows, cols, indptr.data(), idx.data(), val.data(), &h));
        return AdaptiveMat(h);
    }
    // CSC arrays in the narrow host form of sb_upload_compact (rows <= 65536): counts >= 255 go to the side list
    static AdaptiveMat from_csc_compact(Context &ctx, uint32_t rows, uint64_t cols, const std::vector<uint64_t> &indptr,
                                        const std::vector<uint32_t> &idx, const std::vector<uint32_t> &val) {
        std::vector<uint16_t> idx16(idx.size());
        std::vector<uint8_t> cnt8(val.size());
        std::vector<uint64_t> big_pos;
        std::vector<uint32_t> big_cnt;
        for (size_t i = 0; i < idx.size(); i++) {
            idx16[i] = (uint16_t)idx[i];
            cnt8[i] = (uint8_t)std::min<uint32_t>(val[i], 255u);
            if (val[i] >= 255u) {
                big_pos.push_back(i);
                big_cnt.push_back(val[i]);
            }
        }
        sb_mat *h = nullptr;
        check(sb_upload_compact(ctx.raw(), rows, cols, indptr.data(), idx16.data(), cnt8.data(), big_pos.size(), big_pos.data(), big_cnt.data(), &h));
        return AdaptiveMat(h);
    }
    // CSC arrays in the packed host form of sb_upload_packed (gene delta byte + count nibble + side lists), built by the
    // library's host encoder (sb_pack_csc_count / sb_pack_csc_fill)
    static AdaptiveMat from_csc_packed(Context &ctx, uint32_t rows, uint64_t cols, const std::vector<uint64_t> &indptr,
                                       const std::vector<uint32_t> &idx, const std::vector<uint32_t> &val, int threads = 0) {
        uint64_t n_esc = 0, n_big = 0;
        check(sb_pack_csc_count(cols, indptr.data(), idx.data(), val.data(), threads, &n_esc, &n_big));
        std::vector<uint8_t> dgene(idx.size()), cnt4((idx.size() + 1) / 2);
        std::vector<uint64_t> esc_pos(n_esc), big_pos(n_big);
        std::vector<uint32_t> esc_gene(n_esc), big_cnt(n_big);
        check(sb_pack_csc_fill(cols, indptr.data(), idx.data(), val.data(), threads, dgene.data(), cnt4.data(), esc_pos.data(), esc_gene.data(),
                               big_pos.data(), big_cnt.data()));
        sb_mat *h = nullptr;
        check(sb_upload_packed(ctx.raw(), rows, cols, indptr.data(), dgene.data(), cnt4.data(), n_esc, esc_pos.data(), esc_gene.data(), n_big,
                               big_pos.data(), big_cnt.data(), &h));
        return AdaptiveMat(h);
    }
    // from_dense (mat.rs:586-609); dense is row-major rows x cols
    static AdaptiveMat from_dense(Context &ctx, uint32_t rows, uint64_t cols, const std::vector<uint32_t> &dense) {
        std::vector<uint64_t> indptr{0};
        std::vector<uint32_t> idx, val;
        for (uint32_t r = 0; r < rows; r++) {
            for (uint64_t c = 0; c < cols; c++)
                if (dense[r * cols + c]) {
                    idx.push_back((uint32_t)c);
                    val.push_back(dense[r * cols + c]);
                }
            indptr.push_back(idx.size());
        }
        return from_csr(ctx, rows, cols, indptr, idx, val);
    }
    AdaptiveMat(AdaptiveMat &&o) noexcept : h_(o.h_) { o.h_ = nullptr; }
    AdaptiveMat &operator=(AdaptiveMat &&o) noexcept {
        std::swap(h_, o.h_);
        return *this;
    }
    ~AdaptiveMat() {
        if (h_) sb_free_mat(h_);
    }
    size_t rows() const { return shape()[0]; }
    size_t cols() const { return shape()[1]; }
    std::array<size_t, 2> shape() const {
        uint32_t m;
        uint64_t n;
        check(sb_mat_shape(h_, &m, &n, nullptr, nullptr));
        return {m, (size_t)n};
    }
    size_t nnz() const {
        uint64_t z;
        check(sb_mat_shape(h_, nullptr, nullptr, nullptr, &z));
        return z;
    }
    // sum_axis::<u32>(Axis(0)): per-barcode totals (mat.rs:377-406)
    std::vector<uint32_t> sum_axis0_u32() const {
        std::vector<uint32_t> out(cols());
        check(sb_cell_totals(h_, out.data()));
        return out;
    }
    // sum_axis(Axis(1)) in u64 (hdf5-io/src/matrix.rs:106-114)
    std::vector<uint64_t> sum_axis1_u64() const {
        std::vector<uint64_t> out(rows());
        check(sb_gene_totals(h_, 0, out.data()));
        return out;
    }
    // mean_var_axis (mat.rs:285-329); size_factors (optional, one per cell): the SizeNormalized view of diff-exp (diff_exp.rs:340-358)
    std::pair<std::vector<double>, std::vector<double>> mean_var_axis(int axis, const std::vector<double> *size_factors = nullptr) const {
        std::vector<double> mean(axis == 0 ? cols() : rows()), var(mean.size());
        check(sb_mean_var_axis(h_, axis, size_factors ? size_factors->data() : nullptr, mean.data(), var.data()));
        return {std::move(mean), std::move(var)};
    }
    // mean_var_rows (mat.rs:332-374)
    std::pair<std::vector<double>, std::vector<double>> mean_var_rows(const std::vector<uint64_t> &cells, const std::vector<double> *size_factors = nullptr) const {
        std::vector<double> mean(rows()), var(rows());
        check(sb_mean_var_rows(h_, cells.data(), cells.size(), size_factors ? size_factors->data() : nullptr, mean.data(), var.data()));
        return {std::move(mean), std::move(var)};
    }
    // sum_rows_dual (mat.rs:484-583), exact u64
    std::pair<std::vector<uint64_t>, std::vector<uint64_t>> sum_rows_dual(const std::vector<uint64_t> &cols1, const std::vector<uint64_t> &cols2) const {
        std::vector<uint64_t> a(rows()), b(rows());
        check(sb_sum_rows_dual(h_, cols1.data(), cols1.size(), cols2.data(), cols2.size(), a.data(), b.data()));
        return {std::move(a), std::move(b)};
    }
    // size_factors (diff-exp/src/diff_exp.rs:314-334) over all cells
    std::vector<double> size_factors() const {
        std::vector<double> out(cols());
        check(sb_size_factors(h_, nullptr, 0, nullptr, out.data()));
        return out;
    }
    Partition partition_on_threshold(double threshold) const { return partition_on_thresholds(true, threshold, true, threshold); }  // mat.rs:766
    // partition_on_thresholds(Option<f64>, Option<f64>) (mat.rs:772-889)
    Partition partition_on_thresholds(bool has_row, double row_thr, bool has_col, double col_thr) const {
        auto sh = shape();
        std::vector<uint64_t> rows(sh[0]), cols(sh[1]);
        uint64_t nr = 0, nc = 0;
        sb_mat *kept = nullptr, *resid = nullptr;
        check(sb_partition(h_, has_row, row_thr, has_col, col_thr, &kept, &resid, rows.data(), &nr, cols.data(), &nc));
        return Partition(AdaptiveMat(kept), AdaptiveMat(resid), std::vector<size_t>(rows.begin(), rows.begin() + nr),
                         std::vector<size_t>(cols.begin(), cols.begin() + nc));
    }
    AdaptiveMat select_rows(const std::vector<uint32_t> &rows) const {  // mat.rs:1040-1071
        sb_mat *h = nullptr;
        check(sb_select_rows(h_, rows.data(), (uint32_t)rows.size(), &h));
        return AdaptiveMat(h);
    }
    AdaptiveMat select_cols(const std::vector<uint64_t> &cols) const {  // mat.rs:1004-1037
        sb_mat *h = nullptr;
        check(sb_select_cols(h_, cols.data(), cols.size(), &h));
        return AdaptiveMat(h);
    }
    sb_mat *raw() const { return h_; }

  private:
    explicit AdaptiveMat(sb_mat *h) : h_(h) {}
    sb_mat *h_ = nullptr;
    friend class LowRankOffset;
};

// LowRankOffset: A = map(counts) + u.v (low_rank_offset.rs:12-16).  Borrows its AdaptiveMat.
class LowRankOffset {
  public:
    explicit LowRankOffset(sb_nmat *h, const AdaptiveMat &m) : h_(h), mat_(&m) {}
    LowRankOffset(LowRankOffset &&o) noexcept : h_(o.h_), mat_(o.mat_) { o.h_ = nullptr; }
    ~LowRankOffset() {
        if (h_) sb_free_nmat(h_);
    }
    size_t rows() const { return mat_->rows(); }
    size_t cols() const { return mat_->cols(); }
    std::array<size_t, 2> shape() const { return mat_->shape(); }
    Array2 to_dense() const {  // :55-57
        Array2 out(rows(), cols());
        check(sb_nmat_to_dense(h_, out.data.data()));
        return out;
    }
    Array2 dot(const Array2 &rhs) const {  // A . rhs  (:68-81)
        if (rhs.rows != cols()) throw Error(SB_ERR_INVALID_ARG, "Dimension mismatch");
        Array2 out(rows(), rhs.cols);
        check(sb_nmat_dot(h_, rhs.data.data(), (uint32_t)rhs.cols, out.data.data()));
        return out;
    }
    Array2 dot_left(const Array2 &lhs) const {  // lhs . A  (:83-96)
        if (lhs.cols != rows()) throw Error(SB_ERR_INVALID_ARG, "Dimension mismatch");
        Array2 out(lhs.rows, cols());
        check(sb_nmat_rdot(h_, lhs.data.data(), (uint32_t)lhs.rows, out.data.data()));
        return out;
    }
    sb_nmat *raw() const { return h_; }

  private:
    sb_nmat *h_ = nullptr;
    const AdaptiveMat *mat_ = nullptr;
};
}  // namespace sqz

namespace normalization {
enum class Normalization {  // normalization.rs:11-28
    CellRanger = SB_NORM_CELLRANGER,
    CellRanger8 = SB_NORM_CELLRANGER8,
    SeuratLog = SB_NORM_SEURATLOG,
    BinomialDeviance = SB_NORM_BINOMIAL_DEVIANCE,
    BinomialPearson = SB_NORM_BINOMIAL_PEARSON,
    WithSizeFactors = SB_NORM_WITH_SIZE_FACTORS,
    LogTransform = SB_NORM_LOG_TRANSFORM
};
enum class LogBase { E = SB_LOG_E, Two = SB_LOG_TWO, Ten = SB_LOG_TEN };  // :105-112
struct FixedPointFormat {                                                    // :181-187
    uint32_t base, exponent;
};

inline Normalization from_str(const std::string &s) {  // impl FromStr (:30-43)
    if (s == "cellranger") return Normalization::CellRanger;
    if (s == "cellranger8") return Normalization::CellRanger8;
    if (s == "seuratlog") return Normalization::SeuratLog;
    if (s == "binomialdeviance") return Normalization::BinomialDeviance;
    if (s == "binomialpearson") return Normalization::BinomialPearson;
    throw Error(SB_ERR_INVALID_ARG, "Normalization not recognized: " + s);
}

// normalize (:46-69): CellRanger, CellRanger8, SeuratLog; the rest is the reference's panic!("not implemented")
inline sqz::LowRankOffset normalize(const sqz::AdaptiveMat &mat, Normalization norm) {
    if (norm != Normalization::CellRanger && norm != Normalization::CellRanger8 && norm != Normalization::SeuratLog)
        throw Error(SB_ERR_INVALID_ARG, "not implemented");
    sb_nmat *h = nullptr;
    check(sb_normalize(mat.raw(), (int)norm, nullptr, &h));
    return sqz::LowRankOffset(h, mat);
}
// normalize_with_size_factor (:72-102)
inline sqz::LowRankOffset normalize_with_size_factor(const sqz::AdaptiveMat &mat, Normalization norm, const std::vector<uint32_t> *size_factors) {
    if (norm == Normalization::BinomialDeviance || norm == Normalization::BinomialPearson) throw Error(SB_ERR_INVALID_ARG, "not implemented");
    const uint32_t *sf = nullptr;
    if (norm == Normalization::WithSizeFactors && size_factors) {
        if (size_factors->size() != mat.cols()) throw Error(SB_ERR_INVALID_ARG, "Size of the size factor and matrix columns dont match.");
        sf = size_factors->data();
    }
    sb_nmat *h = nullptr;
    check(sb_normalize(mat.raw(), (int)norm, sf, &h));
    return sqz::LowRankOffset(h, mat);
}
// log_normalize_with_size_factor (:138-178): umi_count_sum = nullptr -> median of the barcode totals
inline sqz::LowRankOffset log_normalize_with_size_factor(const sqz::AdaptiveMat &mat, const double *umi_count_sum, LogBase base,
                                                         const std::vector<uint32_t> *size_factors) {
    if (size_factors && size_factors->size() != mat.cols()) throw Error(SB_ERR_INVALID_ARG, "Size of the size factor and matrix columns dont match.");
    sb_nmat *h = nullptr;
    check(sb_log_normalize(mat.raw(), umi_count_sum != nullptr, umi_count_sum ? *umi_count_sum : 0.0, (int)base,
                           size_factors ? size_factors->data() : nullptr, 0, nullptr, &h));
    return sqz::LowRankOffset(h, mat);
}
inline sqz::LowRankOffset log1p_normalize_fixed_point(const sqz::AdaptiveMat &mat, LogBase base, FixedPointFormat fp) {  // :191-213
    sb_nmat *h = nullptr;
    check(sb_normalize_fixed_point(mat.raw(), (int)base, fp.base, fp.exponent, &h));
    return sqz::LowRankOffset(h, mat);
}
inline sqz::LowRankOffset binom_deviance_resid(const sqz::AdaptiveMat &mat) {  // :233-260
    sb_nmat *h = nullptr;
    check(sb_normalize(mat.raw(), SB_NORM_BINOMIAL_DEVIANCE, nullptr, &h));
    return sqz::LowRankOffset(h, mat);
}
inline sqz::LowRankOffset binom_pearson_resid(const sqz::AdaptiveMat &mat) {  // :307-323
    sb_nmat *h = nullptr;
    check(sb_normalize(mat.raw(), SB_NORM_BINOMIAL_PEARSON, nullptr, &h));
    return sqz::LowRankOffset(h, mat);
}
}  // namespace normalization

namespace dim_red {
// PcaResult = (Array2<f64>, Array1<f64>, Array2<f64>) = (u m x k, s k, v n x k)  (dim_red/mod.rs:47)
struct PcaResult {
    Array2 u;
    std::vector<double> s;
    Array2 v;
};

// trait Pca<T, f64> (dim_red/mod.rs:103-111)
struct Pca {
    virtual ~Pca() {}
    virtual PcaResult run_pca_cancellable(const sqz::LowRankOffset &matrix, size_t k, snoop::CancelProgress &c) const = 0;
    PcaResult run_pca(const sqz::LowRankOffset &matrix, size_t k) const {
        snoop::NoOpSnoop s;
        return run_pca_cancellable(matrix, k, s);
    }
};

// svd_bk (bk_svd.rs:57-146); returns (U, sigma, Va) with Va = k x n like the reference
inline std::tuple<Array2, std::vector<double>, Array2> svd_bk(const sqz::LowRankOffset &A, size_t k, size_t b, size_t n_iter, uint64_t seed,
                                                               snoop::CancelProgress &snoop_) {
    Array2 U(A.rows(), k), V(A.cols(), k);
    std::vector<double> S(k);
    check(sb_bksvd(A.raw(), (uint32_t)k, (uint32_t)b, (uint32_t)n_iter, seed, nullptr, snoop::trampoline, &snoop_, U.data.data(), S.data(), V.data.data()));
    Array2 Va(k, A.cols());
    for (size_t c = 0; c < V.rows; c++)
        for (size_t j = 0; j < k; j++) Va(j, c) = V(c, j);
    return {std::move(U), std::move(S), std::move(Va)};
}

struct BkSvd : Pca {  // bk_svd.rs:16-53
    double k_multiplier = 2.0;
    size_t n_iter = 5;
    PcaResult run_pca_cancellable(const sqz::LowRankOffset &array, size_t k, snoop::CancelProgress &c) const override {
        PcaResult r{Array2(array.rows(), k), std::vector<double>(k), Array2(array.cols(), k)};
        check(sb_bksvd_run_pca(array.raw(), (uint32_t)k, k_multiplier, (uint32_t)n_iter, snoop::trampoline, &c, r.u.data.data(), r.s.data(),
                               r.v.data.data()));
        return r;
    }
};

struct RandSvd : Pca {  // rand_svd.rs:13-50 (ignores the snoop, :44-45)
    double l_multiplier = 10.0;
    size_t n_iter = 2;
    PcaResult run_pca_cancellable(const sqz::LowRankOffset &array, size_t k, snoop::CancelProgress &) const override {
        PcaResult r{Array2(array.rows(), k), std::vector<double>(k), Array2(array.cols(), k)};
        check(sb_randsvd_run_pca(array.raw(), (uint32_t)k, l_multiplier, (uint32_t)n_iter, r.u.data.data(), r.s.data(), r.v.data.data()));
        return r;
    }
};

struct Irlba : Pca {  // irlba.rs:36-69 (the reference cannot run it on a LowRankOffset: no 1-D Dot; the device type can)
    double tol = 0.0001;
    size_t max_iter = 50;
    PcaResult run_pca_cancellable(const sqz::LowRankOffset &array, size_t k, snoop::CancelProgress &c) const override {
        PcaResult r{Array2(array.rows(), k), std::vector<double>(k), Array2(array.cols(), k)};
        check(sb_irlba(array.raw(), (uint32_t)k, tol, (uint32_t)max_iter, nullptr, snoop::trampoline, &c, r.u.data.data(), r.s.data(), r.v.data.data(),
                       nullptr, nullptr));
        return r;
    }
};

// frobenius (dim_red/mod.rs:114-122): sqrt(sum v^2) / (rows * cols)
inline double frobenius(const Array2 &a) {
    double acc = 0.0;
    for (double v : a.data) acc += v * v;
    return std::sqrt(acc) / (double)(a.rows * a.cols);
}
}  // namespace dim_red

// diff-exp: sSeq (compute_sseq_params, sseq_differential_expression; the contract is stated in scanb200.h)
namespace diff_exp {
struct SSeqParams {
    uint64_t num_cells = 0;
    uint32_t num_genes = 0;
    std::vector<double> size_factors;  // this rank's cells
    std::vector<double> gene_means, gene_variances;
    std::vector<uint8_t> use_genes;
    std::vector<double> gene_moment_phi;
    double zeta_hat = 0.0, delta = 0.0;
    std::vector<double> gene_phi;
};
struct DiffExpResult {
    std::vector<uint8_t> genes_tested;
    std::vector<uint64_t> sums_in, sums_out;
    std::vector<double> common_mean, common_dispersion;
    std::vector<double> normalized_mean_in, normalized_mean_out;
    std::vector<double> p_values, adjusted_p_values, log2_fold_change;
};

inline SSeqParams compute_sseq_params(const sqz::AdaptiveMat &mat, double zeta_quantile = 0.995) {
    const size_t m = mat.rows();
    SSeqParams p;
    p.size_factors.resize(mat.cols());
    p.gene_means.resize(m);
    p.gene_variances.resize(m);
    p.use_genes.resize(m);
    p.gene_moment_phi.resize(m);
    p.gene_phi.resize(m);
    sb_sseq_params c{0, 0, 0, 0.0, 0.0, p.size_factors.data(), p.gene_means.data(), p.gene_variances.data(), p.gene_moment_phi.data(),
                     p.gene_phi.data(), p.use_genes.data()};
    check(sb_sseq_compute_params(mat.raw(), zeta_quantile, &c));
    p.num_cells = c.num_cells;
    p.num_genes = c.num_genes;
    p.zeta_hat = c.zeta_hat;
    p.delta = c.delta;
    return p;
}

namespace detail {
// the C view of the params: the library only reads them
inline sb_sseq_params view(const SSeqParams &p) {
    return sb_sseq_params{p.num_cells, p.num_genes, 0, p.zeta_hat, p.delta, const_cast<double *>(p.size_factors.data()),
                          const_cast<double *>(p.gene_means.data()), const_cast<double *>(p.gene_variances.data()),
                          const_cast<double *>(p.gene_moment_phi.data()), const_cast<double *>(p.gene_phi.data()),
                          const_cast<uint8_t *>(p.use_genes.data())};
}
template <class F>
std::vector<DiffExpResult> run(const SSeqParams &p, size_t n_comp, size_t m, F call) {
    std::vector<uint64_t> s_in(n_comp * m), s_out(n_comp * m);
    std::vector<double> nm_in(n_comp * m), nm_out(n_comp * m), pv(n_comp * m), q(n_comp * m), lfc(n_comp * m);
    sb_diff_exp_out o{s_in.data(), s_out.data(), nm_in.data(), nm_out.data(), pv.data(), q.data(), lfc.data()};
    sb_sseq_params c = view(p);
    check(call(&c, &o));
    std::vector<DiffExpResult> out(n_comp);
    for (size_t j = 0; j < n_comp; j++) {
        auto sl = [&](const auto &v) { return std::vector<typename std::decay_t<decltype(v)>::value_type>(v.begin() + j * m, v.begin() + (j + 1) * m); };
        out[j] = DiffExpResult{p.use_genes, sl(s_in), sl(s_out), p.gene_means, p.gene_phi, sl(nm_in), sl(nm_out), sl(pv), sl(q), sl(lfc)};
    }
    return out;
}
}  // namespace detail

// cond_in / cond_out: strictly ascending (local) cell indices
inline DiffExpResult sseq_differential_expression(const sqz::AdaptiveMat &mat, const std::vector<uint64_t> &cond_in, const std::vector<uint64_t> &cond_out,
                                                  const SSeqParams &params, uint64_t big_count = 900) {
    return detail::run(params, 1, mat.rows(), [&](const sb_sseq_params *c, sb_diff_exp_out *o) {
        return sb_sseq_diff_exp(mat.raw(), c, cond_in.data(), cond_in.size(), cond_out.data(), cond_out.size(), big_count, o);
    })[0];
}
// one result per group j: cells labelled j against all others
inline std::vector<DiffExpResult> sseq_one_vs_rest(const sqz::AdaptiveMat &mat, const std::vector<uint32_t> &labels, uint32_t n_groups,
                                                   const SSeqParams &params, uint64_t big_count = 900) {
    if (labels.size() != mat.cols()) throw Error(SB_ERR_INVALID_ARG, "one label per cell");
    return detail::run(params, n_groups, mat.rows(), [&](const sb_sseq_params *c, sb_diff_exp_out *o) {
        return sb_sseq_one_vs_rest(mat.raw(), c, labels.data(), n_groups, big_count, o);
    });
}
// one result per pair (a, b): cells labelled a against cells labelled b, one matrix pass for all pairs
inline std::vector<DiffExpResult> sseq_pairs(const sqz::AdaptiveMat &mat, const std::vector<uint32_t> &labels, uint32_t n_groups,
                                             const std::vector<std::pair<uint32_t, uint32_t>> &pairs, const SSeqParams &params, uint64_t big_count = 900) {
    if (labels.size() != mat.cols()) throw Error(SB_ERR_INVALID_ARG, "one label per cell");
    std::vector<uint32_t> flat;
    for (const auto &p : pairs) {
        flat.push_back(p.first);
        flat.push_back(p.second);
    }
    return detail::run(params, pairs.size(), mat.rows(), [&](const sb_sseq_params *c, sb_diff_exp_out *o) {
        return sb_sseq_pairs(mat.raw(), c, labels.data(), n_groups, flat.data(), (uint32_t)pairs.size(), big_count, o);
    });
}
}  // namespace diff_exp

// graph clustering: SNN graph of the kNN lists and deterministic Louvain (the rules are stated in scanb200.h)
namespace clustering {
struct Graph {  // symmetric CSR, weights = Jaccard index << 24
    std::vector<uint64_t> indptr;
    std::vector<uint32_t> indices;
    std::vector<uint64_t> weights;
};
struct Options {
    double resolution = 1.0;
    uint32_t max_levels = SB_LOUVAIN_MAX_LEVELS;
    uint32_t max_iterations = 100;
};
struct Level {
    uint64_t nodes;
    uint32_t iterations;
    double modularity;
};
struct Result {
    std::vector<uint32_t> labels;  // 0..n_clusters-1, by size, descending
    uint32_t n_clusters = 0;
    double modularity = 0.0;
    std::vector<Level> levels;
};

namespace detail {
inline Result result(std::vector<uint32_t> labels, const sb_louvain_info &info) {
    Result r{std::move(labels), info.n_clusters, info.modularity, {}};
    for (uint32_t l = 0; l < info.n_levels; l++) r.levels.push_back(Level{info.level_nodes[l], info.level_iterations[l], info.level_modularity[l]});
    return r;
}
inline sb_louvain_opts opts(const Options &o) { return sb_louvain_opts{o.resolution, o.max_levels, o.max_iterations}; }
}  // namespace detail

// nbr: n x k row-major, as knn returns it
inline Graph snn_graph(const Context &ctx, const std::vector<uint32_t> &nbr, uint32_t k) {
    if (k == 0 || nbr.size() % k) throw Error(SB_ERR_INVALID_ARG, "nbr must hold n x k entries");
    const uint64_t n = nbr.size() / k;
    Graph g{std::vector<uint64_t>(n + 1), std::vector<uint32_t>(2 * n * k), std::vector<uint64_t>(2 * n * k)};
    uint64_t nnz = 0;
    check(sb_snn_graph(ctx.raw(), nbr.data(), n, k, g.indptr.data(), g.indices.data(), g.weights.data(), &nnz));
    g.indices.resize(nnz);
    g.weights.resize(nnz);
    return g;
}
inline Result louvain(const Context &ctx, const Graph &g, const Options &o = Options()) {
    if (g.indptr.empty()) throw Error(SB_ERR_INVALID_ARG, "indptr must hold n + 1 entries");
    const uint64_t n = g.indptr.size() - 1;
    std::vector<uint32_t> labels(n);
    sb_louvain_info info;
    const sb_louvain_opts c = detail::opts(o);
    check(sb_louvain(ctx.raw(), n, g.indptr.data(), g.indices.data(), g.weights.data(), &c, labels.data(), &info));
    return detail::result(std::move(labels), info);
}
// on a sharded context: this rank's rows (global indices) -> this rank's labels
inline Result cluster_knn(const Context &ctx, const std::vector<uint32_t> &nbr, uint32_t k, const Options &o = Options()) {
    if (k == 0 || nbr.size() % k) throw Error(SB_ERR_INVALID_ARG, "nbr must hold n x k entries");
    const uint64_t n = nbr.size() / k;
    std::vector<uint32_t> labels(n);
    sb_louvain_info info;
    const sb_louvain_opts c = detail::opts(o);
    check(sb_cluster_knn(ctx.raw(), nbr.data(), n, k, &c, labels.data(), &info));
    return detail::result(std::move(labels), info);
}

// complete linkage (NN-chain) of points [n x dim] on the host: Z [(n - 1) x 4] in scipy's layout
inline std::vector<double> linkage_complete(const std::vector<double> &points, uint32_t dim) {
    if (dim == 0 || points.size() % dim) throw Error(SB_ERR_INVALID_ARG, "points must hold n x dim entries");
    const uint32_t n = (uint32_t)(points.size() / dim);
    std::vector<double> Z((n > 1 ? n - 1 : 0) * 4);
    check(sb_linkage_complete(points.data(), n, dim, Z.data()));
    return Z;
}
struct MergeOptions {
    double adj_p_threshold = 0.05;
    uint32_t min_de_genes = 1;
    uint64_t big_count = 900;
};
struct MergeResult {
    std::vector<uint32_t> labels;  // 0..n_clusters-1, by size, descending
    uint32_t n_clusters = 0, n_rounds = 0;
    uint64_t pairs_tested = 0, pairs_merged = 0;
};
// Cell Ranger's MERGE_CLUSTERS: scores [n_local x dim] (the PCA scores), labels of this rank's cells
inline MergeResult merge_clusters(const sqz::AdaptiveMat &mat, const diff_exp::SSeqParams &params, const std::vector<double> &scores, uint32_t dim,
                                  const std::vector<uint32_t> &labels, uint32_t n_groups, const MergeOptions &o = MergeOptions()) {
    if (labels.size() != mat.cols() || scores.size() != labels.size() * dim) throw Error(SB_ERR_INVALID_ARG, "one label and one score row per cell");
    MergeResult r;
    r.labels.resize(labels.size());
    const sb_merge_opts c{o.adj_p_threshold, o.min_de_genes, 0, o.big_count};
    const sb_sseq_params p = diff_exp::detail::view(params);
    sb_merge_info info;
    check(sb_merge_clusters(mat.raw(), &p, scores.data(), dim, labels.data(), n_groups, &c, r.labels.data(), &info));
    r.n_clusters = info.n_clusters;
    r.n_rounds = info.n_rounds;
    r.pairs_tested = info.pairs_tested;
    r.pairs_merged = info.pairs_merged;
    return r;
}
}  // namespace clustering

// UMAP embedding: fuzzy kNN graph and epoch-synchronous layout (the rules are stated in scanb200.h)
namespace embedding {
struct Graph {  // symmetric CSR, weights in (0, 1]
    std::vector<uint64_t> indptr;
    std::vector<uint32_t> indices;
    std::vector<double> weights;
    std::vector<double> rho, sigma;  // per vertex (from umap_graph)
};
enum class Init : uint32_t { Pca = SB_UMAP_INIT_PCA, Random = SB_UMAP_INIT_RANDOM, User = SB_UMAP_INIT_USER };
struct Options {
    uint32_t n_components = 2;
    uint32_t n_epochs = 0;  // 0: 500 if n <= 10,000 else 200
    double min_dist = 0.1, spread = 1.0;
    double a = 0.0, b = 0.0;  // both 0: fitted
    double learning_rate = 1.0, repulsion_strength = 1.0, set_op_mix_ratio = 1.0;
    uint32_t negative_sample_rate = 5;
    Init init = Init::Pca;
    uint64_t seed = 0;
};
struct Result {
    std::vector<double> embedding;  // n x n_components, row-major
    double a = 0.0, b = 0.0, max_weight = 0.0;
    uint32_t n_epochs = 0;
    uint64_t n_edges = 0, n_edges_used = 0;
};

namespace detail {
inline sb_umap_opts opts(const Options &o) {
    return sb_umap_opts{o.n_components, o.n_epochs, o.min_dist, o.spread, o.a, o.b, o.learning_rate, o.repulsion_strength, o.set_op_mix_ratio,
                        o.negative_sample_rate, (uint32_t)o.init, o.seed};
}
inline Result result(std::vector<double> emb, const sb_umap_info &info) {
    return Result{std::move(emb), info.a, info.b, info.max_weight, info.n_epochs, info.n_edges, info.n_edges_used};
}
inline uint64_t rows(const std::vector<double> &scores, uint32_t dim, const std::vector<uint32_t> &nbr, uint32_t k) {
    if (dim == 0 || scores.size() % dim) throw Error(SB_ERR_INVALID_ARG, "scores must hold n x dim entries");
    if (k == 0 || nbr.size() != scores.size() / dim * k) throw Error(SB_ERR_INVALID_ARG, "nbr must hold n x k entries");
    return scores.size() / dim;
}
}  // namespace detail

// scores: n x dim, nbr: n x k row-major, as knn returns it
inline Graph umap_graph(const Context &ctx, const std::vector<double> &scores, uint32_t dim, const std::vector<uint32_t> &nbr, uint32_t k,
                        const Options &o = Options()) {
    const uint64_t n = detail::rows(scores, dim, nbr, k);
    Graph g{std::vector<uint64_t>(n + 1), std::vector<uint32_t>(2 * n * k), std::vector<double>(2 * n * k), std::vector<double>(n), std::vector<double>(n)};
    uint64_t nnz = 0;
    const sb_umap_opts c = detail::opts(o);
    check(sb_umap_graph(ctx.raw(), scores.data(), nbr.data(), n, dim, k, &c, g.indptr.data(), g.indices.data(), g.weights.data(), &nnz, g.rho.data(),
                        g.sigma.data()));
    g.indices.resize(nnz);
    g.weights.resize(nnz);
    return g;
}
// init: n x n_components (scaled per column with Init::Pca, as given with Init::User, unused with Init::Random)
inline Result umap_layout(const Context &ctx, const Graph &g, const std::vector<double> &init, const Options &o = Options()) {
    if (g.indptr.empty()) throw Error(SB_ERR_INVALID_ARG, "indptr must hold n + 1 entries");
    const uint64_t n = g.indptr.size() - 1;
    if (o.init != Init::Random && init.size() != n * o.n_components) throw Error(SB_ERR_INVALID_ARG, "init must hold n x n_components entries");
    std::vector<double> out(n * o.n_components);
    sb_umap_info info;
    const sb_umap_opts c = detail::opts(o);
    check(sb_umap_layout(ctx.raw(), n, g.indptr.data(), g.indices.data(), g.weights.data(), init.empty() ? nullptr : init.data(), &c, out.data(), &info));
    return detail::result(std::move(out), info);
}
// on a sharded context: this rank's rows (global neighbour indices) -> this rank's rows of the embedding
inline Result umap(const Context &ctx, const std::vector<double> &scores, uint32_t dim, const std::vector<uint32_t> &nbr, uint32_t k,
                   const Options &o = Options(), const std::vector<double> &init = {}) {
    const uint64_t n = detail::rows(scores, dim, nbr, k);
    if (o.init == Init::User && init.size() != n * o.n_components) throw Error(SB_ERR_INVALID_ARG, "init must hold n x n_components entries");
    std::vector<double> out(n * o.n_components);
    sb_umap_info info;
    const sb_umap_opts c = detail::opts(o);
    check(sb_umap(ctx.raw(), scores.data(), nbr.data(), n, dim, k, &c, init.empty() ? nullptr : init.data(), out.data(), &info));
    return detail::result(std::move(out), info);
}
// t-SNE embedding: perplexity-calibrated affinities and a deterministic Barnes-Hut layout (the rules are stated in scanb200.h)
struct Affinities {  // symmetric P as a CSR, entries in (0, 1] summing to 1
    std::vector<uint64_t> indptr;
    std::vector<uint32_t> indices;
    std::vector<double> P;
    std::vector<double> beta;  // per point (from tsne_affinities)
};
enum class TsneInit : uint32_t { Pca = SB_TSNE_INIT_PCA, Random = SB_TSNE_INIT_RANDOM, User = SB_TSNE_INIT_USER };
struct TsneOptions {  // bhtsne's names and defaults
    double perplexity = 30.0;
    double theta = 0.5;             // 0: the exact gradient
    double learning_rate = 200.0;   // 0: max(n / (4 early_exaggeration), 50)
    double early_exaggeration = 12.0;
    uint32_t max_iter = 1000, stop_lying_iter = 250, mom_switch_iter = 250;
    TsneInit init = TsneInit::Pca;
    uint64_t seed = 0;
};
struct TsneResult {
    std::vector<double> embedding;  // n x 2, row-major
    double kl_divergence = 0.0, learning_rate = 0.0;
    uint64_t nnz = 0;
    uint32_t n_iter = 0;
};

namespace detail {
inline sb_tsne_opts tsne_opts(const TsneOptions &o) {
    return sb_tsne_opts{o.perplexity, o.theta, o.learning_rate, o.early_exaggeration, o.max_iter, o.stop_lying_iter, o.mom_switch_iter, 2,
                        (uint32_t)o.init, 0, o.seed};
}
inline TsneResult tsne_result(std::vector<double> emb, const sb_tsne_info &info) {
    return TsneResult{std::move(emb), info.kl_divergence, info.learning_rate, info.nnz, info.n_iter};
}
}  // namespace detail

// scores: n x dim, nbr: n x k row-major, as knn returns it (k = min(n - 1, floor(3 perplexity)))
inline Affinities tsne_affinities(const Context &ctx, const std::vector<double> &scores, uint32_t dim, const std::vector<uint32_t> &nbr, uint32_t k,
                                  const TsneOptions &o = TsneOptions()) {
    const uint64_t n = detail::rows(scores, dim, nbr, k);
    Affinities a{std::vector<uint64_t>(n + 1), std::vector<uint32_t>(2 * n * k), std::vector<double>(2 * n * k), std::vector<double>(n)};
    uint64_t nnz = 0;
    const sb_tsne_opts c = detail::tsne_opts(o);
    check(sb_tsne_affinities(ctx.raw(), scores.data(), nbr.data(), n, dim, k, &c, a.indptr.data(), a.indices.data(), a.P.data(), &nnz, a.beta.data()));
    a.indices.resize(nnz);
    a.P.resize(nnz);
    return a;
}
// init: n x 2 (the first two score columns with TsneInit::Pca, as given with TsneInit::User, unused with TsneInit::Random)
inline TsneResult tsne_layout(const Context &ctx, const Affinities &a, const std::vector<double> &init, const TsneOptions &o = TsneOptions()) {
    if (a.indptr.empty()) throw Error(SB_ERR_INVALID_ARG, "indptr must hold n + 1 entries");
    const uint64_t n = a.indptr.size() - 1;
    if (o.init != TsneInit::Random && init.size() != n * 2) throw Error(SB_ERR_INVALID_ARG, "init must hold n x 2 entries");
    std::vector<double> out(n * 2);
    sb_tsne_info info;
    const sb_tsne_opts c = detail::tsne_opts(o);
    check(sb_tsne_layout(ctx.raw(), n, a.indptr.data(), a.indices.data(), a.P.data(), init.empty() ? nullptr : init.data(), &c, out.data(), &info));
    return detail::tsne_result(std::move(out), info);
}
// on a sharded context: this rank's rows (global neighbour indices) -> this rank's rows of the embedding
inline TsneResult tsne(const Context &ctx, const std::vector<double> &scores, uint32_t dim, const std::vector<uint32_t> &nbr, uint32_t k,
                       const TsneOptions &o = TsneOptions(), const std::vector<double> &init = {}) {
    const uint64_t n = detail::rows(scores, dim, nbr, k);
    if (o.init == TsneInit::User && init.size() != n * 2) throw Error(SB_ERR_INVALID_ARG, "init must hold n x 2 entries");
    std::vector<double> out(n * 2);
    sb_tsne_info info;
    const sb_tsne_opts c = detail::tsne_opts(o);
    check(sb_tsne(ctx.raw(), scores.data(), nbr.data(), n, dim, k, &c, init.empty() ? nullptr : init.data(), out.data(), &info));
    return detail::tsne_result(std::move(out), info);
}
}  // namespace embedding
}  // namespace scanb200
