"""scan_rs_b200 -- B200-native normalize -> PCA hot path of scan-rs behind a C ABI.

The package mirrors the reference's module layout for this path only:
  sqz            AdaptiveMat (device-resident counts), LowRankOffset (normalized matrix)
  normalization  Normalization, normalize, normalize_with_size_factor, ...
  dim_red        BkSvd, RandSvd, Irlba, svd_bk, svd_rand, irlba
  snoop          NoOpSnoop, AtomicSnoop
  mtx            load_mtx (gz MatrixMarket -> device matrix)
  nn             knn, find_nn on the PCA scores
  cluster        SNN graph of the kNN lists and deterministic Louvain (snn_graph, louvain, cluster_knn); merging of over-split
                 clusters by differential expression (linkage_complete, merge_clusters)
  embedding      UMAP of the scores and kNN lists: fuzzy graph and deterministic layout (umap_graph, umap_layout, umap); t-SNE:
                 perplexity-calibrated affinities and a deterministic Barnes-Hut layout (tsne_affinities, tsne_layout, tsne)
  diff_exp       sSeq differential expression (compute_sseq_params, sseq_differential_expression, sseq_one_vs_rest, sseq_pairs)
  synth          synthetic workloads (test / bench utility)
All compute runs in scan_rs_b200/libscanb200.so (hand-written sm_100a CUDA + cuSOLVER/cuBLAS for the
small dense steps); there is no CPU fallback."""
from ._lib import CancellationError, ScanB200Error, LIB_PATH  # noqa: F401
from .sqz import AdaptiveMat, Context, LowRankOffset  # noqa: F401
from .normalization import (LogBase, Normalization, binom_deviance_resid, binom_pearson_resid,  # noqa: F401
                            log1p_normalize_fixed_point, log_normalize, log_normalize_with_size_factor,
                            normalize, normalize_with_size_factor)
from .dim_red import BkSvd, Irlba, RandSvd, irlba, irlba_start, omega, pinned_outputs, svd_bk, svd_rand, variance_explained  # noqa: F401
ScanError = ScanB200Error
from .snoop import AtomicSnoop, NoOpSnoop  # noqa: F401
from .mtx import load_mtx  # noqa: F401
from .nn import find_nn, knn  # noqa: F401
from .multi import MultiContext  # noqa: F401
from .diff_exp import (DiffExpResult, SSeqParams, compute_sseq_params, sseq_differential_expression,  # noqa: F401
                       sseq_one_vs_rest, sseq_pairs)
from .cluster import (ClusterResult, LouvainOptions, MergeOptions, MergeResult, cluster_knn, linkage_complete, louvain,  # noqa: F401
                      merge_clusters, snn_graph)
from .embedding import (TsneOptions, TsneResult, UmapOptions, UmapResult, tsne, tsne_affinities, tsne_layout, umap, umap_graph,  # noqa: F401
                        umap_layout)
