"""reid_gan_b200 -- B200-native (sm_100a) drop-in for the pseudo-label hot path of
cluster-contrast-reid as found in daemon-219/ReID-GAN:

  compute_jaccard_distance   clustercontrast/utils/faiss_rerank.py:30
  DBSCAN                     sklearn.cluster.DBSCAN as called at examples/cluster_contrast_train_usl.py:160,163
  generate_cluster_features  examples/cluster_contrast_train_usl.py:169-182 (+ F.normalize :191)
  ClusterMemory, cm, cm_hard clustercontrast/models/cm.py:36,75,110-137
  DistributedClusterMemory   ClusterMemory of nn.DataParallel's concatenated batch, one process per GPU
  Evaluator, evaluate_all    clustercontrast/evaluators.py:91-142, device-resident; re_ranking_features re-ranks from features
  DistributedEvaluator       Evaluator of nn.DataParallel's evaluation, one process per GPU (eval_shard splits the images)

Python/PyTorch host code over a C-ABI CUDA library (include/reid_b200.h); no faiss, no Triton, no
backend dispatch and no CPU fallback: importing works anywhere, calling needs a B200.
"""
from .faiss_rerank import compute_jaccard_distance, JaccardDistance, rerank_state, knn_search  # noqa: F401
from .dbscan import DBSCAN  # noqa: F401
from .centroids import generate_cluster_features  # noqa: F401
from .cm import CM, CM_Hard, cm, cm_hard, ClusterMemory  # noqa: F401
from .cm_dist import DistributedClusterMemory  # noqa: F401
from .rerank import re_ranking, re_ranking_features  # noqa: F401
from .evaluation import pairwise_distance, mean_ap, cmc  # noqa: F401
from .infomap_cluster import get_dist_nbr, get_links  # noqa: F401
from .synth import synth, synth_cm_batch, synth_device, synth_hard  # noqa: F401
from . import pipeline  # noqa: F401
from .evaluators import DeviceFeatures, extract_features, shard_items, eval_shard, Evaluator, evaluate_all  # noqa: F401
from .eval_dist import DistributedEvaluator  # noqa: F401

__all__ = ["pairwise_distance", "mean_ap", "cmc", "re_ranking", "re_ranking_features", "Evaluator", "DistributedEvaluator", "eval_shard", "evaluate_all", "get_dist_nbr", "get_links", "compute_jaccard_distance", "JaccardDistance", "DBSCAN", "generate_cluster_features",
           "CM", "CM_Hard", "cm", "cm_hard", "ClusterMemory", "DistributedClusterMemory", "synth", "synth_cm_batch"]
