//! scan-b200 -- the normalize -> PCA hot path of scan-rs on B200 GPUs, behind the reference's own entry points.
//!
//! Call sites change from (tools/src/bin/cmd.rs:67-81)
//! ```ignore
//! let norm_mat = normalize(matrix.view(), normalization);
//! let (u, d, v) = BkSvd::new().run_pca(&norm_mat, num_pcs)?;
//! ```
//! to
//! ```ignore
//! let ctx = scan_b200::Context::new(0)?;
//! let dev = scan_b200::DeviceCountMatrix::upload(&ctx, &matrix.view())?;
//! let norm_mat = dev.normalize(normalization, None)?;              // impl DataMat
//! let (u, d, v) = scan_b200::GpuBkSvd::new().run_pca(&norm_mat, num_pcs)?;   // the same PcaResult
//! ```
//! The normalized matrix of the reference is `LowRankOffset<D, impl MatrixMap<u32, f64>>` (normalization.rs:46): the map is an
//! opaque closure chain a backend cannot introspect, so the device path owns both steps and takes the UN-normalized matrix.
//!
//! NOT COMPILED where it was written (no rustc in that image).  The C ABI underneath is exercised by the C++ layer
//! (include/scanb200.hpp, tests/cpp/host_api_test.cpp) and the Python layer (scan_rs_b200/*.py); `src/ffi.rs` is generated from
//! include/scanb200.h.
pub mod ffi;

use anyhow::{format_err, Error};
use ndarray::{Array1, Array2};
use scan_rs::dim_red::{DataMat, Pca, PcaResult};
use scan_rs::normalization::Normalization;
use snoop::{CancelProgress, CancellationError};
use sqz::{AdaptiveMat, AdaptiveVec, MatrixMap};
use std::ffi::{c_void, CStr};
use std::marker::PhantomData;
use std::ops::Deref;

fn check(rc: i32) -> Result<(), Error> {
    if rc == ffi::SB_OK {
        return Ok(());
    }
    if rc == ffi::SB_ERR_CANCELLED {
        return Err(CancellationError.into()); // snoop/src/lib.rs:5-18
    }
    let msg = unsafe { CStr::from_ptr(ffi::sb_last_error()) }.to_string_lossy().into_owned();
    Err(format_err!("{msg}")) // "The input matrix must be at least 2x2." / "invalid k" verbatim (bk_svd.rs:74,78)
}

/// One GPU + stream.  `!Send`: a context is driven from the thread that uses it (SURVEY 8b).
pub struct Context {
    h: *mut ffi::sb_ctx,
    owned: bool,
}

impl Context {
    pub fn new(device: i32) -> Result<Self, Error> {
        let mut h = std::ptr::null_mut();
        check(unsafe { ffi::sb_init(device, &mut h) })?; // no CPU fallback: SB_ERR_CUDA without a device
        Ok(Self { h, owned: true })
    }
    pub fn set_option(&self, name: &str, value: f64) -> Result<(), Error> {
        let c = std::ffi::CString::new(name)?;
        check(unsafe { ffi::sb_set_option(self.h, c.as_ptr(), value) })
    }
}
impl Drop for Context {
    fn drop(&mut self) {
        if self.owned {
            unsafe { ffi::sb_shutdown(self.h) }
        }
    }
}

/// `AdaptiveMat<u32>` resident on the device (cell-major + the layouts both products stream).
pub struct DeviceCountMatrix<'c> {
    h: *mut ffi::sb_mat,
    rows: usize,
    cols: usize,
    _ctx: PhantomData<&'c Context>,
}

impl<'c> DeviceCountMatrix<'c> {
    /// Decode every AdaptiveVec once (`foreach`, vec.rs:1230-1273) into u64 indptr / u32 index / u32 count and upload.
    pub fn upload<D, M>(ctx: &'c Context, mat: &AdaptiveMat<u32, D, M>) -> Result<Self, Error>
    where
        D: Deref<Target = [AdaptiveVec]>,
        M: MatrixMap<u32, u32>,
    {
        let (mut indptr, mut idx, mut val) = (vec![0u64], Vec::<u32>::new(), Vec::<u32>::new());
        for (i, v) in mat.iter().enumerate() {
            // rows if CSR, columns if CSC (mat.rs:178-187)
            v.foreach(|j, x| {
                let x = mat.get_map().map(x, i, j);
                if x != 0 {
                    idx.push(j as u32);
                    val.push(x);
                }
            });
            indptr.push(idx.len() as u64);
        }
        let major = if mat.is_csr() { ffi::SB_GENE_MAJOR } else { ffi::SB_CELL_MAJOR };
        let mut h = std::ptr::null_mut();
        check(unsafe {
            ffi::sb_upload(ctx.h, major, mat.rows() as u32, mat.cols() as u64, indptr.as_ptr(), idx.as_ptr(), val.as_ptr(), &mut h)
        })?;
        Ok(Self { h, rows: mat.rows(), cols: mat.cols(), _ctx: PhantomData })
    }

    /// The same walk into the narrow host form (cell-major, at most 65,536 genes): u16 gene + u8 count, counts >= 255 in a side
    /// list -- 3 bytes per entry cross PCIe instead of 8, and the copy is the largest part of an end-to-end call.
    pub fn upload_compact<D, M>(ctx: &'c Context, mat: &AdaptiveMat<u32, D, M>) -> Result<Self, Error>
    where
        D: Deref<Target = [AdaptiveVec]>,
        M: MatrixMap<u32, u32>,
    {
        assert!(!mat.is_csr() && mat.rows() <= 65536);
        let (mut indptr, mut idx, mut cnt) = (vec![0u64], Vec::<u16>::new(), Vec::<u8>::new());
        let (mut big_pos, mut big_cnt) = (Vec::<u64>::new(), Vec::<u32>::new());
        for (c, v) in mat.iter().enumerate() {
            v.foreach(|g, x| {
                let x = mat.get_map().map(x, g, c);
                if x != 0 {
                    if x >= 255 {
                        big_pos.push(idx.len() as u64);
                        big_cnt.push(x);
                    }
                    idx.push(g as u16);
                    cnt.push(x.min(255) as u8);
                }
            });
            indptr.push(idx.len() as u64);
        }
        let mut h = std::ptr::null_mut();
        check(unsafe {
            ffi::sb_upload_compact(ctx.h, mat.rows() as u32, mat.cols() as u64, indptr.as_ptr(), idx.as_ptr(), cnt.as_ptr(),
                                   big_pos.len() as u64, big_pos.as_ptr(), big_cnt.as_ptr(), &mut h)
        })?;
        Ok(Self { h, rows: mat.rows(), cols: mat.cols(), _ctx: PhantomData })
    }

    /// The same walk into the packed host form (cell-major, any gene count): one byte of gene delta + one nibble of count per
    /// entry, escapes in two side lists -- about 1.6 bytes per entry cross PCIe (the compact form: 3, the plain one: 8).  The
    /// layout is stated beside `sb_upload_packed` in include/scanb200.h; `sb_pack_csc_fill` builds it from plain arrays.
    pub fn upload_packed<D, M>(ctx: &'c Context, mat: &AdaptiveMat<u32, D, M>) -> Result<Self, Error>
    where
        D: Deref<Target = [AdaptiveVec]>,
        M: MatrixMap<u32, u32>,
    {
        assert!(!mat.is_csr());
        let (mut indptr, mut dgene, mut cnt4) = (vec![0u64], Vec::<u8>::new(), Vec::<u8>::new());
        let (mut esc_pos, mut esc_gene) = (Vec::<u64>::new(), Vec::<u32>::new());
        let (mut big_pos, mut big_cnt) = (Vec::<u64>::new(), Vec::<u32>::new());
        for (c, v) in mat.iter().enumerate() {
            let mut prev: i64 = -1;
            v.foreach(|g, x| {
                let x = mat.get_map().map(x, g, c);
                if x != 0 {
                    let pos = dgene.len() as u64;
                    let d = g as i64 - prev;
                    if d >= 1 && d <= 255 {
                        dgene.push(d as u8);
                    } else {
                        dgene.push(0);
                        esc_pos.push(pos);
                        esc_gene.push(g as u32);
                    }
                    let nib = if x >= 15 {
                        big_pos.push(pos);
                        big_cnt.push(x);
                        15u8
                    } else {
                        x as u8
                    };
                    if pos % 2 == 0 {
                        cnt4.push(nib);
                    } else {
                        *cnt4.last_mut().unwrap() |= nib << 4;
                    }
                    prev = g as i64;
                }
            });
            indptr.push(dgene.len() as u64);
        }
        let mut h = std::ptr::null_mut();
        check(unsafe {
            ffi::sb_upload_packed(ctx.h, mat.rows() as u32, mat.cols() as u64, indptr.as_ptr(), dgene.as_ptr(), cnt4.as_ptr(),
                                  esc_pos.len() as u64, esc_pos.as_ptr(), esc_gene.as_ptr(),
                                  big_pos.len() as u64, big_pos.as_ptr(), big_cnt.as_ptr(), &mut h)
        })?;
        Ok(Self { h, rows: mat.rows(), cols: mat.cols(), _ctx: PhantomData })
    }

    pub fn shape(&self) -> [usize; 2] {
        [self.rows, self.cols]
    }

    /// sum_axis::<u32>(Axis(0)) (mat.rs:377-406): per-cell UMI totals
    pub fn cell_totals(&self) -> Result<Array1<u32>, Error> {
        let mut out = Array1::<u32>::zeros(self.cols);
        check(unsafe { ffi::sb_cell_totals(self.h, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// normalize / normalize_with_size_factor (normalization.rs:46-102); the enum order is SB_NORM_*
    pub fn normalize(&self, norm: Normalization, size_factors: Option<&Array1<u32>>) -> Result<DeviceNormalized<'_>, Error> {
        let mut h = std::ptr::null_mut();
        let sf = size_factors.map_or(std::ptr::null(), |a| a.as_ptr());
        check(unsafe { ffi::sb_normalize(self.h, norm as i32, sf, &mut h) })?;
        Ok(DeviceNormalized { h, mat: self })
    }

    /// mean_var_axis(Axis(1)) of the SizeNormalized view (diff-exp/src/diff_exp.rs:458-472)
    pub fn mean_var_genes(&self, size_factors: Option<&[f64]>) -> Result<(Array1<f64>, Array1<f64>), Error> {
        let (mut mean, mut var) = (Array1::<f64>::zeros(self.rows), Array1::<f64>::zeros(self.rows));
        let sf = size_factors.map_or(std::ptr::null(), |a| a.as_ptr());
        check(unsafe { ffi::sb_mean_var_axis(self.h, 1, sf, mean.as_mut_ptr(), var.as_mut_ptr()) })?;
        Ok((mean, var))
    }
}
impl Drop for DeviceCountMatrix<'_> {
    fn drop(&mut self) {
        unsafe { ffi::sb_free_mat(self.h) }
    }
}

/// `LowRankOffset<D, impl MatrixMap<u32, f64>>` on the device: counts + fused map + rank-1 offset, never materialised.
pub struct DeviceNormalized<'a> {
    h: *mut ffi::sb_nmat,
    mat: &'a DeviceCountMatrix<'a>,
}
impl DataMat for DeviceNormalized<'_> {
    fn shape(&self) -> [usize; 2] {
        self.mat.shape()
    }
}
impl Drop for DeviceNormalized<'_> {
    fn drop(&mut self) {
        unsafe { ffi::sb_free_nmat(self.h) } // before the matrix it borrows: guaranteed by the lifetime
    }
}

unsafe extern "C" fn progress_trampoline<S: CancelProgress>(fraction: f64, user: *mut c_void) -> i32 {
    let s = &mut *(user as *mut S);
    s.set_progress_check(fraction).is_err() as i32 // Err(CancellationError) -> stop at this milestone
}

/// A local struct (not `BkSvd`): the blanket `impl<T> Pca<T, f64> for BkSvd` (bk_svd.rs:41-47) must not be overlapped.
pub struct GpuBkSvd {
    pub k_multiplier: f64,
    pub n_iter: usize,
}
impl GpuBkSvd {
    pub fn new() -> Self {
        Self { k_multiplier: 2.0, n_iter: 5 } // BkSvd::new (bk_svd.rs:24-31)
    }
}
impl Default for GpuBkSvd {
    fn default() -> Self {
        Self::new()
    }
}
impl<'a> Pca<DeviceNormalized<'a>, f64> for GpuBkSvd {
    fn run_pca_cancellable(&self, a: &DeviceNormalized<'a>, k: usize, mut snoop: impl CancelProgress) -> Result<PcaResult, Error> {
        let [m, n] = a.shape();
        let (mut u, mut s, mut v) = (Array2::<f64>::zeros((m, k)), Array1::<f64>::zeros(k), Array2::<f64>::zeros((n, k)));
        check(unsafe {
            ffi::sb_bksvd_run_pca(a.h, k as u32, self.k_multiplier, self.n_iter as u32, Some(progress_trampoline::<_>),
                                  &mut snoop as *mut _ as *mut c_void, u.as_mut_ptr(), s.as_mut_ptr(), v.as_mut_ptr())
        })?;
        Ok((u, s, v)) // v is already vt.reversed_axes() (bk_svd.rs:51)
    }
}

/// RandSvd (rand_svd.rs:13-50): ignores the snoop, as the reference does.
pub struct GpuRandSvd {
    pub l_multiplier: f64,
    pub n_iter: usize,
}
impl GpuRandSvd {
    pub fn new() -> Self {
        Self { l_multiplier: 10.0, n_iter: 2 }
    }
}
impl<'a> Pca<DeviceNormalized<'a>, f64> for GpuRandSvd {
    fn run_pca_cancellable(&self, a: &DeviceNormalized<'a>, k: usize, _snoop: impl CancelProgress) -> Result<PcaResult, Error> {
        let [m, n] = a.shape();
        let (mut u, mut s, mut v) = (Array2::<f64>::zeros((m, k)), Array1::<f64>::zeros(k), Array2::<f64>::zeros((n, k)));
        check(unsafe {
            ffi::sb_randsvd_run_pca(a.h, k as u32, self.l_multiplier, self.n_iter as u32, u.as_mut_ptr(), s.as_mut_ptr(), v.as_mut_ptr())
        })?;
        Ok((u, s, v))
    }
}

/// Irlba (irlba.rs:36-69).  The reference cannot run IRLBA on a LowRankOffset (no 1-D `Dot`); the device type can.
pub struct GpuIrlba {
    pub tol: f64,
    pub max_iter: usize,
}
impl GpuIrlba {
    pub fn new() -> Self {
        Self { tol: 0.0001, max_iter: 50 }
    }
}
impl<'a> Pca<DeviceNormalized<'a>, f64> for GpuIrlba {
    fn run_pca_cancellable(&self, a: &DeviceNormalized<'a>, k: usize, mut snoop: impl CancelProgress) -> Result<PcaResult, Error> {
        let [m, n] = a.shape();
        let (mut u, mut s, mut v) = (Array2::<f64>::zeros((m, k)), Array1::<f64>::zeros(k), Array2::<f64>::zeros((n, k)));
        check(unsafe {
            ffi::sb_irlba(a.h, k as u32, self.tol, self.max_iter as u32, std::ptr::null(), Some(progress_trampoline::<_>),
                          &mut snoop as *mut _ as *mut c_void, u.as_mut_ptr(), s.as_mut_ptr(), v.as_mut_ptr(),
                          std::ptr::null_mut(), std::ptr::null_mut())
        })?;
        Ok((u, s, v))
    }
}

/// diff-exp's `SSeqParams` (compute_sseq_params): the per-gene moments of the size-normalized view and the shrunken dispersions.
/// `size_factors` holds this rank's cells; the gene arrays are replicated.
#[derive(Clone, Debug)]
pub struct SSeqParams {
    pub num_cells: usize,
    pub num_genes: usize,
    pub size_factors: Array1<f64>,
    pub gene_means: Array1<f64>,
    pub gene_variances: Array1<f64>,
    pub use_genes: Array1<bool>,
    pub gene_moment_phi: Array1<f64>,
    pub zeta_hat: f64,
    pub delta: f64,
    pub gene_phi: Array1<f64>,
}

/// diff-exp's `DiffExpResult` for one comparison.
#[derive(Clone, Debug)]
pub struct DiffExpResult {
    pub genes_tested: Array1<bool>,
    pub sums_in: Array1<u64>,
    pub sums_out: Array1<u64>,
    pub common_mean: Array1<f64>,
    pub common_dispersion: Array1<f64>,
    pub normalized_mean_in: Array1<f64>,
    pub normalized_mean_out: Array1<f64>,
    pub p_values: Array1<f64>,
    pub adjusted_p_values: Array1<f64>,
    pub log2_fold_change: Array1<f64>,
}

/// compute_sseq_params on the device (the contract is stated beside `sb_sseq_compute_params` in include/scanb200.h)
pub fn compute_sseq_params(mat: &DeviceCountMatrix<'_>, zeta_quantile: f64) -> Result<SSeqParams, Error> {
    let [m, n] = mat.shape();
    let (mut sf, mut mean, mut var) = (Array1::<f64>::zeros(n), Array1::<f64>::zeros(m), Array1::<f64>::zeros(m));
    let (mut phi_mm, mut phi, mut use_g) = (Array1::<f64>::zeros(m), Array1::<f64>::zeros(m), Array1::<u8>::zeros(m));
    let mut p = ffi::sb_sseq_params {
        num_cells: 0, num_genes: 0, reserved: 0, zeta_hat: 0.0, delta: 0.0, size_factors: sf.as_mut_ptr(), gene_means: mean.as_mut_ptr(),
        gene_variances: var.as_mut_ptr(), gene_moment_phi: phi_mm.as_mut_ptr(), gene_phi: phi.as_mut_ptr(), use_genes: use_g.as_mut_ptr(),
    };
    check(unsafe { ffi::sb_sseq_compute_params(mat.h, zeta_quantile, &mut p) })?;
    Ok(SSeqParams {
        num_cells: p.num_cells as usize, num_genes: p.num_genes as usize, size_factors: sf, gene_means: mean, gene_variances: var,
        use_genes: use_g.mapv(|u| u != 0), gene_moment_phi: phi_mm, zeta_hat: p.zeta_hat, delta: p.delta, gene_phi: phi,
    })
}

fn sseq_run(mat: &DeviceCountMatrix<'_>, params: &SSeqParams, n_comp: usize,
            call: impl FnOnce(*const ffi::sb_sseq_params, *mut ffi::sb_diff_exp_out) -> i32) -> Result<Vec<DiffExpResult>, Error> {
    let m = mat.shape()[0];
    let (mut s_in, mut s_out) = (Array2::<u64>::zeros((n_comp, m)), Array2::<u64>::zeros((n_comp, m)));
    let mut f: Vec<Array2<f64>> = (0..5).map(|_| Array2::<f64>::zeros((n_comp, m))).collect();
    // the library only reads the params; the C struct carries mutable pointers because sb_sseq_compute_params fills the same type
    let (mut sf, mut mean, mut var, mut phi_mm, mut phi) = (params.size_factors.to_owned(), params.gene_means.to_owned(),
        params.gene_variances.to_owned(), params.gene_moment_phi.to_owned(), params.gene_phi.to_owned());
    let mut use_g = params.use_genes.mapv(|b| b as u8);
    let p = ffi::sb_sseq_params {
        num_cells: params.num_cells as u64, num_genes: params.num_genes as u32, reserved: 0, zeta_hat: params.zeta_hat, delta: params.delta,
        size_factors: sf.as_mut_ptr(), gene_means: mean.as_mut_ptr(), gene_variances: var.as_mut_ptr(), gene_moment_phi: phi_mm.as_mut_ptr(),
        gene_phi: phi.as_mut_ptr(), use_genes: use_g.as_mut_ptr(),
    };
    let mut o = ffi::sb_diff_exp_out {
        sums_in: s_in.as_mut_ptr(), sums_out: s_out.as_mut_ptr(), normalized_mean_in: f[0].as_mut_ptr(), normalized_mean_out: f[1].as_mut_ptr(),
        p_values: f[2].as_mut_ptr(), adjusted_p_values: f[3].as_mut_ptr(), log2_fold_change: f[4].as_mut_ptr(),
    };
    check(call(&p, &mut o))?;
    Ok((0..n_comp)
        .map(|j| DiffExpResult {
            genes_tested: params.use_genes.clone(),
            sums_in: s_in.row(j).to_owned(),
            sums_out: s_out.row(j).to_owned(),
            common_mean: params.gene_means.clone(),
            common_dispersion: params.gene_phi.clone(),
            normalized_mean_in: f[0].row(j).to_owned(),
            normalized_mean_out: f[1].row(j).to_owned(),
            p_values: f[2].row(j).to_owned(),
            adjusted_p_values: f[3].row(j).to_owned(),
            log2_fold_change: f[4].row(j).to_owned(),
        })
        .collect())
}

/// sseq_differential_expression: `cond_in` against `cond_out` (strictly ascending local cell indices)
pub fn sseq_differential_expression(mat: &DeviceCountMatrix<'_>, cond_in: &[u64], cond_out: &[u64], params: &SSeqParams, big_count: u64)
                                    -> Result<DiffExpResult, Error> {
    let mut r = sseq_run(mat, params, 1, |p, o| unsafe {
        ffi::sb_sseq_diff_exp(mat.h, p, cond_in.as_ptr(), cond_in.len() as u64, cond_out.as_ptr(), cond_out.len() as u64, big_count, o)
    })?;
    Ok(r.remove(0))
}

/// Cell Ranger's cluster-vs-rest loop, batched: result j compares the cells labelled j with all other cells
pub fn sseq_one_vs_rest(mat: &DeviceCountMatrix<'_>, labels: &[u32], n_groups: u32, params: &SSeqParams, big_count: u64)
                        -> Result<Vec<DiffExpResult>, Error> {
    assert_eq!(labels.len(), mat.shape()[1], "one label per cell");
    sseq_run(mat, params, n_groups as usize, |p, o| unsafe { ffi::sb_sseq_one_vs_rest(mat.h, p, labels.as_ptr(), n_groups, big_count, o) })
}

/// Pairwise comparisons, batched: result j compares the cells labelled `pairs[j].0` with the cells labelled `pairs[j].1`, bit for
/// bit what `sseq_differential_expression` gives with those cells, in one pass over the matrix
pub fn sseq_pairs(mat: &DeviceCountMatrix<'_>, labels: &[u32], n_groups: u32, pairs: &[(u32, u32)], params: &SSeqParams, big_count: u64)
                  -> Result<Vec<DiffExpResult>, Error> {
    assert_eq!(labels.len(), mat.shape()[1], "one label per cell");
    let flat: Vec<u32> = pairs.iter().flat_map(|&(a, b)| [a, b]).collect();
    sseq_run(mat, params, pairs.len(), |p, o| unsafe {
        ffi::sb_sseq_pairs(mat.h, p, labels.as_ptr(), n_groups, flat.as_ptr(), pairs.len() as u32, big_count, o)
    })
}

/// Louvain options: resolution (gamma) > 0, max_levels 1..32, max_iterations per level >= 1
#[derive(Clone, Copy, Debug)]
pub struct LouvainOptions {
    pub resolution: f64,
    pub max_levels: u32,
    pub max_iterations: u32,
}
impl Default for LouvainOptions {
    fn default() -> Self {
        LouvainOptions { resolution: 1.0, max_levels: ffi::SB_LOUVAIN_MAX_LEVELS as u32, max_iterations: 100 }
    }
}

/// Cluster labels (0..n_clusters-1, by size, descending), the final modularity and (nodes, iterations, Q) per level
#[derive(Clone, Debug)]
pub struct Clustering {
    pub labels: Vec<u32>,
    pub n_clusters: u32,
    pub modularity: f64,
    pub levels: Vec<(u64, u32, f64)>,
}

/// Shared-nearest-neighbour graph as a symmetric CSR; weights are Jaccard indices in 24-bit fixed point
#[derive(Clone, Debug)]
pub struct SnnGraph {
    pub indptr: Vec<u64>,
    pub indices: Vec<u32>,
    pub weights: Vec<u64>,
}

fn clustering(labels: Vec<u32>, info: &ffi::sb_louvain_info) -> Clustering {
    let levels = (0..info.n_levels as usize).map(|l| (info.level_nodes[l], info.level_iterations[l], info.level_modularity[l])).collect();
    Clustering { labels, n_clusters: info.n_clusters, modularity: info.modularity, levels }
}
fn louvain_opts(o: &LouvainOptions) -> ffi::sb_louvain_opts {
    ffi::sb_louvain_opts { resolution: o.resolution, max_levels: o.max_levels, max_iterations: o.max_iterations }
}
fn empty_info() -> ffi::sb_louvain_info {
    ffi::sb_louvain_info { n_clusters: 0, n_levels: 0, modularity: 0.0, level_nodes: [0; ffi::SB_LOUVAIN_MAX_LEVELS],
                           level_iterations: [0; ffi::SB_LOUVAIN_MAX_LEVELS], level_modularity: [0.0; ffi::SB_LOUVAIN_MAX_LEVELS] }
}

/// The SNN graph of kNN lists (`nbr` n x k, as `knn` returns them; the rules are stated beside `sb_snn_graph` in include/scanb200.h)
pub fn snn_graph(ctx: &Context, nbr: &Array2<u32>) -> Result<SnnGraph, Error> {
    let nbr = nbr.as_standard_layout();
    let (n, k) = nbr.dim();
    let mut g = SnnGraph { indptr: vec![0; n + 1], indices: vec![0; 2 * n * k], weights: vec![0; 2 * n * k] };
    let mut nnz = 0u64;
    check(unsafe {
        ffi::sb_snn_graph(ctx.h, nbr.as_ptr(), n as u64, k as u32, g.indptr.as_mut_ptr(), g.indices.as_mut_ptr(), g.weights.as_mut_ptr(), &mut nnz)
    })?;
    g.indices.truncate(nnz as usize);
    g.weights.truncate(nnz as usize);
    Ok(g)
}

/// Deterministic Louvain on a symmetric CSR with integer weights
pub fn louvain(ctx: &Context, g: &SnnGraph, opts: &LouvainOptions) -> Result<Clustering, Error> {
    assert!(!g.indptr.is_empty(), "indptr must hold n + 1 entries");
    let n = g.indptr.len() - 1;
    let mut labels = vec![0u32; n];
    let mut info = empty_info();
    let o = louvain_opts(opts);
    check(unsafe { ffi::sb_louvain(ctx.h, n as u64, g.indptr.as_ptr(), g.indices.as_ptr(), g.weights.as_ptr(), &o, labels.as_mut_ptr(), &mut info) })?;
    Ok(clustering(labels, &info))
}

/// kNN lists -> SNN graph -> Louvain with the graph kept on the device; on a sharded context every rank passes its own rows
/// (global indices) and receives its own cells' labels
pub fn cluster_knn(ctx: &Context, nbr: &Array2<u32>, opts: &LouvainOptions) -> Result<Clustering, Error> {
    let nbr = nbr.as_standard_layout();
    let (n, k) = nbr.dim();
    let mut labels = vec![0u32; n];
    let mut info = empty_info();
    let o = louvain_opts(opts);
    check(unsafe { ffi::sb_cluster_knn(ctx.h, nbr.as_ptr(), n as u64, k as u32, &o, labels.as_mut_ptr(), &mut info) })?;
    Ok(clustering(labels, &info))
}

/// Complete linkage (NN-chain) of `points` (n x dim) on the host: Z ((n - 1) x 4) in scipy's layout
pub fn linkage_complete(points: &Array2<f64>) -> Result<Array2<f64>, Error> {
    let pts = points.as_standard_layout();
    let (n, dim) = pts.dim();
    let mut z = Array2::<f64>::zeros((n.saturating_sub(1), 4));
    check(unsafe { ffi::sb_linkage_complete(pts.as_ptr(), n as u32, dim as u32, z.as_mut_ptr()) })?;
    Ok(z)
}

/// Cluster-merge options: a pair merges when fewer than `min_de_genes` genes have adjusted p below `adj_p_threshold`
#[derive(Clone, Copy, Debug)]
pub struct MergeOptions {
    pub adj_p_threshold: f64,
    pub min_de_genes: u32,
    pub big_count: u64,
}
impl Default for MergeOptions {
    fn default() -> Self {
        MergeOptions { adj_p_threshold: 0.05, min_de_genes: 1, big_count: 900 }
    }
}

/// Merged labels (0..n_clusters-1, by size, descending), rounds, sibling pairs tested and merged
#[derive(Clone, Debug)]
pub struct MergeResult {
    pub labels: Vec<u32>,
    pub n_clusters: u32,
    pub n_rounds: u32,
    pub pairs_tested: u64,
    pub pairs_merged: u64,
}

/// Cell Ranger's MERGE_CLUSTERS (the rule is stated beside `sb_merge_clusters` in include/scanb200.h): `scores` are the PCA scores
/// of this rank's cells, `labels` their clusters (each < n_groups)
pub fn merge_clusters(mat: &DeviceCountMatrix<'_>, params: &SSeqParams, scores: &Array2<f64>, labels: &[u32], n_groups: u32, opts: &MergeOptions)
                      -> Result<MergeResult, Error> {
    let sc = scores.as_standard_layout();
    assert_eq!(labels.len(), mat.shape()[1], "one label per cell");
    assert_eq!(sc.nrows(), labels.len(), "one score row per cell");
    let mut out = vec![0u32; labels.len()];
    let mut info = ffi::sb_merge_info { n_clusters: 0, n_rounds: 0, pairs_tested: 0, pairs_merged: 0 };
    let o = ffi::sb_merge_opts { adj_p_threshold: opts.adj_p_threshold, min_de_genes: opts.min_de_genes, reserved: 0, big_count: opts.big_count };
    // the library only reads the params (see sseq_run)
    let (mut sf, mut mean, mut var, mut phi_mm, mut phi) = (params.size_factors.to_owned(), params.gene_means.to_owned(),
        params.gene_variances.to_owned(), params.gene_moment_phi.to_owned(), params.gene_phi.to_owned());
    let mut use_g = params.use_genes.mapv(|b| b as u8);
    let p = ffi::sb_sseq_params {
        num_cells: params.num_cells as u64, num_genes: params.num_genes as u32, reserved: 0, zeta_hat: params.zeta_hat, delta: params.delta,
        size_factors: sf.as_mut_ptr(), gene_means: mean.as_mut_ptr(), gene_variances: var.as_mut_ptr(), gene_moment_phi: phi_mm.as_mut_ptr(),
        gene_phi: phi.as_mut_ptr(), use_genes: use_g.as_mut_ptr(),
    };
    check(unsafe {
        ffi::sb_merge_clusters(mat.h, &p, sc.as_ptr(), sc.ncols() as u32, labels.as_ptr(), n_groups, &o, out.as_mut_ptr(), &mut info)
    })?;
    Ok(MergeResult { labels: out, n_clusters: info.n_clusters, n_rounds: info.n_rounds, pairs_tested: info.pairs_tested, pairs_merged: info.pairs_merged })
}

/// How the UMAP layout starts: the first score columns scaled to [0, 10], the counter hash, or the caller's positions
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum UmapInit {
    Pca,
    Random,
    User,
}

/// UMAP options (umap-learn's names and defaults; n_epochs 0: 500 up to 10,000 cells, else 200; a = b = 0: fitted)
#[derive(Clone, Copy, Debug)]
pub struct UmapOptions {
    pub n_components: u32,
    pub n_epochs: u32,
    pub min_dist: f64,
    pub spread: f64,
    pub a: f64,
    pub b: f64,
    pub learning_rate: f64,
    pub repulsion_strength: f64,
    pub set_op_mix_ratio: f64,
    pub negative_sample_rate: u32,
    pub init: UmapInit,
    pub seed: u64,
}
impl Default for UmapOptions {
    fn default() -> Self {
        UmapOptions { n_components: 2, n_epochs: 0, min_dist: 0.1, spread: 1.0, a: 0.0, b: 0.0, learning_rate: 1.0, repulsion_strength: 1.0,
                      set_op_mix_ratio: 1.0, negative_sample_rate: 5, init: UmapInit::Pca, seed: 0 }
    }
}

/// The fuzzy kNN graph as a symmetric CSR (weights in (0, 1]) with every vertex's rho and sigma
#[derive(Clone, Debug)]
pub struct UmapGraph {
    pub indptr: Vec<u64>,
    pub indices: Vec<u32>,
    pub weights: Vec<f64>,
    pub rho: Vec<f64>,
    pub sigma: Vec<f64>,
}

/// The embedding (n x n_components) and the layout's parameters as used
#[derive(Clone, Debug)]
pub struct Umap {
    pub embedding: Array2<f64>,
    pub a: f64,
    pub b: f64,
    pub n_epochs: u32,
    pub n_edges: u64,
    pub n_edges_used: u64,
    pub max_weight: f64,
}

fn umap_opts(o: &UmapOptions) -> ffi::sb_umap_opts {
    let init = match o.init {
        UmapInit::Pca => ffi::SB_UMAP_INIT_PCA,
        UmapInit::Random => ffi::SB_UMAP_INIT_RANDOM,
        UmapInit::User => ffi::SB_UMAP_INIT_USER,
    };
    ffi::sb_umap_opts { n_components: o.n_components, n_epochs: o.n_epochs, min_dist: o.min_dist, spread: o.spread, a: o.a, b: o.b,
                        learning_rate: o.learning_rate, repulsion_strength: o.repulsion_strength, set_op_mix_ratio: o.set_op_mix_ratio,
                        negative_sample_rate: o.negative_sample_rate, init, seed: o.seed }
}
fn umap_result(out: Vec<f64>, n: usize, nc: usize, info: &ffi::sb_umap_info) -> Umap {
    Umap { embedding: Array2::from_shape_vec((n, nc), out).expect("n x n_components"), a: info.a, b: info.b, n_epochs: info.n_epochs,
           n_edges: info.n_edges, n_edges_used: info.n_edges_used, max_weight: info.max_weight }
}
fn empty_umap_info() -> ffi::sb_umap_info {
    ffi::sb_umap_info { a: 0.0, b: 0.0, max_weight: 0.0, n_edges: 0, n_edges_used: 0, n_epochs: 0 }
}

/// The fuzzy kNN graph of the scores (n x dim) and their kNN lists (n x k, as `knn` returns them; the rules are stated beside
/// `sb_umap_graph` in include/scanb200.h)
pub fn umap_graph(ctx: &Context, scores: &Array2<f64>, nbr: &Array2<u32>, opts: &UmapOptions) -> Result<UmapGraph, Error> {
    let scores = scores.as_standard_layout();
    let nbr = nbr.as_standard_layout();
    let ((n, dim), k) = (scores.dim(), nbr.dim().1);
    assert_eq!(nbr.dim().0, n, "scores and nbr must have the same rows");
    let mut g = UmapGraph { indptr: vec![0; n + 1], indices: vec![0; 2 * n * k], weights: vec![0.0; 2 * n * k], rho: vec![0.0; n], sigma: vec![0.0; n] };
    let mut nnz = 0u64;
    let o = umap_opts(opts);
    check(unsafe {
        ffi::sb_umap_graph(ctx.h, scores.as_ptr(), nbr.as_ptr(), n as u64, dim as u32, k as u32, &o, g.indptr.as_mut_ptr(), g.indices.as_mut_ptr(),
                           g.weights.as_mut_ptr(), &mut nnz, g.rho.as_mut_ptr(), g.sigma.as_mut_ptr())
    })?;
    g.indices.truncate(nnz as usize);
    g.weights.truncate(nnz as usize);
    Ok(g)
}

/// The layout of a symmetric CSR; `init` (n x n_components) is scaled per column with `UmapInit::Pca`, taken as given with
/// `UmapInit::User` and not read with `UmapInit::Random`
pub fn umap_layout(ctx: &Context, g: &UmapGraph, init: Option<&Array2<f64>>, opts: &UmapOptions) -> Result<Umap, Error> {
    assert!(!g.indptr.is_empty(), "indptr must hold n + 1 entries");
    let (n, nc) = (g.indptr.len() - 1, opts.n_components as usize);
    let init = init.map(|a| a.as_standard_layout().into_owned());
    if let Some(a) = &init {
        assert_eq!(a.dim(), (n, nc), "init must be n x n_components");
    }
    let mut out = vec![0.0; n * nc];
    let mut info = empty_umap_info();
    let o = umap_opts(opts);
    let ip = init.as_ref().map_or(std::ptr::null(), |a| a.as_ptr());
    check(unsafe { ffi::sb_umap_layout(ctx.h, n as u64, g.indptr.as_ptr(), g.indices.as_ptr(), g.weights.as_ptr(), ip, &o, out.as_mut_ptr(), &mut info) })?;
    Ok(umap_result(out, n, nc, &info))
}

/// Scores and kNN lists -> fuzzy graph -> layout with the graph kept on the device; on a sharded context every rank passes its own
/// rows (global neighbour indices) and receives its own rows of the embedding
pub fn umap(ctx: &Context, scores: &Array2<f64>, nbr: &Array2<u32>, opts: &UmapOptions, init: Option<&Array2<f64>>) -> Result<Umap, Error> {
    let scores = scores.as_standard_layout();
    let nbr = nbr.as_standard_layout();
    let ((n, dim), k, nc) = (scores.dim(), nbr.dim().1, opts.n_components as usize);
    assert_eq!(nbr.dim().0, n, "scores and nbr must have the same rows");
    let init = init.map(|a| a.as_standard_layout().into_owned());
    if let Some(a) = &init {
        assert_eq!(a.dim(), (n, nc), "init must be n x n_components");
    }
    let mut out = vec![0.0; n * nc];
    let mut info = empty_umap_info();
    let o = umap_opts(opts);
    let ip = init.as_ref().map_or(std::ptr::null(), |a| a.as_ptr());
    check(unsafe { ffi::sb_umap(ctx.h, scores.as_ptr(), nbr.as_ptr(), n as u64, dim as u32, k as u32, &o, ip, out.as_mut_ptr(), &mut info) })?;
    Ok(umap_result(out, n, nc, &info))
}

/// Start of the t-SNE layout
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum TsneInit {
    Pca,
    Random,
    User,
}

/// t-SNE options (bhtsne's names and defaults; learning_rate 0: max(n / (4 early_exaggeration), 50); 2 components)
#[derive(Clone, Copy, Debug)]
pub struct TsneOptions {
    pub perplexity: f64,
    pub theta: f64,
    pub learning_rate: f64,
    pub early_exaggeration: f64,
    pub max_iter: u32,
    pub stop_lying_iter: u32,
    pub mom_switch_iter: u32,
    pub init: TsneInit,
    pub seed: u64,
}
impl Default for TsneOptions {
    fn default() -> Self {
        TsneOptions { perplexity: 30.0, theta: 0.5, learning_rate: 200.0, early_exaggeration: 12.0, max_iter: 1000, stop_lying_iter: 250,
                      mom_switch_iter: 250, init: TsneInit::Pca, seed: 0 }
    }
}

/// The symmetric affinities P as a CSR (entries in (0, 1], summing to 1) with every point's beta
#[derive(Clone, Debug)]
pub struct TsneAffinities {
    pub indptr: Vec<u64>,
    pub indices: Vec<u32>,
    pub p: Vec<f64>,
    pub beta: Vec<f64>,
}

/// The embedding (n x 2) and the layout's summary
#[derive(Clone, Debug)]
pub struct Tsne {
    pub embedding: Array2<f64>,
    pub kl_divergence: f64,
    pub learning_rate: f64,
    pub nnz: u64,
    pub n_iter: u32,
}

fn tsne_opts(o: &TsneOptions) -> ffi::sb_tsne_opts {
    let init = match o.init {
        TsneInit::Pca => ffi::SB_TSNE_INIT_PCA,
        TsneInit::Random => ffi::SB_TSNE_INIT_RANDOM,
        TsneInit::User => ffi::SB_TSNE_INIT_USER,
    };
    ffi::sb_tsne_opts { perplexity: o.perplexity, theta: o.theta, learning_rate: o.learning_rate, early_exaggeration: o.early_exaggeration,
                        max_iter: o.max_iter, stop_lying_iter: o.stop_lying_iter, mom_switch_iter: o.mom_switch_iter, n_components: 2, init,
                        reserved: 0, seed: o.seed }
}
fn tsne_result(out: Vec<f64>, n: usize, info: &ffi::sb_tsne_info) -> Tsne {
    Tsne { embedding: Array2::from_shape_vec((n, 2), out).expect("n x 2"), kl_divergence: info.kl_divergence, learning_rate: info.learning_rate,
           nnz: info.nnz, n_iter: info.n_iter }
}
fn empty_tsne_info() -> ffi::sb_tsne_info {
    ffi::sb_tsne_info { kl_divergence: 0.0, learning_rate: 0.0, nnz: 0, n_iter: 0, reserved: 0 }
}

/// The t-SNE affinities of the scores (n x dim) and their kNN lists (n x k with k = min(n - 1, floor(3 perplexity)), as `knn`
/// returns them; the rules are stated beside `sb_tsne_affinities` in include/scanb200.h)
pub fn tsne_affinities(ctx: &Context, scores: &Array2<f64>, nbr: &Array2<u32>, opts: &TsneOptions) -> Result<TsneAffinities, Error> {
    let scores = scores.as_standard_layout();
    let nbr = nbr.as_standard_layout();
    let ((n, dim), k) = (scores.dim(), nbr.dim().1);
    assert_eq!(nbr.dim().0, n, "scores and nbr must have the same rows");
    let mut a = TsneAffinities { indptr: vec![0; n + 1], indices: vec![0; 2 * n * k], p: vec![0.0; 2 * n * k], beta: vec![0.0; n] };
    let mut nnz = 0u64;
    let o = tsne_opts(opts);
    check(unsafe {
        ffi::sb_tsne_affinities(ctx.h, scores.as_ptr(), nbr.as_ptr(), n as u64, dim as u32, k as u32, &o, a.indptr.as_mut_ptr(), a.indices.as_mut_ptr(),
                                a.p.as_mut_ptr(), &mut nnz, a.beta.as_mut_ptr())
    })?;
    a.indices.truncate(nnz as usize);
    a.p.truncate(nnz as usize);
    Ok(a)
}

/// The t-SNE layout of P from `init` (n x 2: the first two score columns with TsneInit::Pca, as given with TsneInit::User, unused
/// with TsneInit::Random)
pub fn tsne_layout(ctx: &Context, a: &TsneAffinities, init: Option<&Array2<f64>>, opts: &TsneOptions) -> Result<Tsne, Error> {
    assert!(!a.indptr.is_empty(), "indptr must hold n + 1 entries");
    let n = a.indptr.len() - 1;
    let init = init.map(|x| x.as_standard_layout().into_owned());
    if let Some(x) = &init {
        assert_eq!(x.dim(), (n, 2), "init must be n x 2");
    }
    let mut out = vec![0.0; n * 2];
    let mut info = empty_tsne_info();
    let o = tsne_opts(opts);
    let ip = init.as_ref().map_or(std::ptr::null(), |x| x.as_ptr());
    check(unsafe { ffi::sb_tsne_layout(ctx.h, n as u64, a.indptr.as_ptr(), a.indices.as_ptr(), a.p.as_ptr(), ip, &o, out.as_mut_ptr(), &mut info) })?;
    Ok(tsne_result(out, n, &info))
}

/// Scores and kNN lists -> affinities -> layout with P kept on the device; on a sharded context every rank passes its own rows
/// (global neighbour indices) and gets its own rows of the embedding
pub fn tsne(ctx: &Context, scores: &Array2<f64>, nbr: &Array2<u32>, opts: &TsneOptions, init: Option<&Array2<f64>>) -> Result<Tsne, Error> {
    let scores = scores.as_standard_layout();
    let nbr = nbr.as_standard_layout();
    let ((n, dim), k) = (scores.dim(), nbr.dim().1);
    assert_eq!(nbr.dim().0, n, "scores and nbr must have the same rows");
    let init = init.map(|x| x.as_standard_layout().into_owned());
    if let Some(x) = &init {
        assert_eq!(x.dim(), (n, 2), "init must be n x 2");
    }
    let mut out = vec![0.0; n * 2];
    let mut info = empty_tsne_info();
    let o = tsne_opts(opts);
    let ip = init.as_ref().map_or(std::ptr::null(), |x| x.as_ptr());
    check(unsafe { ffi::sb_tsne(ctx.h, scores.as_ptr(), nbr.as_ptr(), n as u64, dim as u32, k as u32, &o, ip, out.as_mut_ptr(), &mut info) })?;
    Ok(tsne_result(out, n, &info))
}

/// Every GPU of the box from one caller thread (SURVEY 8b; the reference's only caller is a single process).  `run` executes the
/// closure once per rank, concurrently, each on its own library worker thread with its own `Context`; inside it a rank uploads
/// its contiguous cell shard and makes the ordinary calls -- the collectives meet across the workers.
pub struct MultiGpu {
    h: *mut ffi::sb_multi,
    n: usize,
}
impl MultiGpu {
    pub fn new(devices: &[i32]) -> Result<Self, Error> {
        let mut h = std::ptr::null_mut();
        check(unsafe { ffi::sb_multi_init(devices.len() as i32, devices.as_ptr(), &mut h) })?;
        Ok(Self { h, n: devices.len() })
    }
    pub fn size(&self) -> usize {
        self.n
    }
    pub fn run<F>(&self, f: F) -> Result<(), Error>
    where
        F: Fn(usize, &Context) -> Result<(), Error> + Sync,
    {
        unsafe extern "C" fn tramp<F: Fn(usize, &Context) -> Result<(), Error> + Sync>(rank: i32, ctx: *mut ffi::sb_ctx, user: *mut c_void) -> i32 {
            let f = &*(user as *const F);
            let c = Context { h: ctx, owned: false };
            match std::panic::catch_unwind(std::panic::AssertUnwindSafe(|| f(rank as usize, &c))) {
                Ok(Ok(())) => ffi::SB_OK,
                Ok(Err(e)) => if e.is::<CancellationError>() { ffi::SB_ERR_CANCELLED } else { ffi::SB_ERR_INVALID_ARG },
                Err(_) => ffi::SB_ERR_INVALID_ARG, // no panic crosses the ABI
            }
        }
        check(unsafe { ffi::sb_multi_run(self.h, Some(tramp::<F>), &f as *const F as *mut c_void) })
    }
}
impl Drop for MultiGpu {
    fn drop(&mut self) {
        unsafe { ffi::sb_multi_shutdown(self.h) }
    }
}
