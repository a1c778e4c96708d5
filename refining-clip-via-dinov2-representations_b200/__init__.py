"""B200-native DINO-Soft loss path (drop-in for the reference's ``open_clip.loss.ClipLossWithDINOEnhancements``).

Import as ``dinosoft_b200`` (see the shim at the repo root).  Contents:

    loss.py      the nn.Module with the reference's ctor/forward signature, gather_features,
                 compute_student_tau, install_into_open_clip
    feature_store.py  device-resident DINO feature store: bf16 table in HBM, gather kernel with on-device range
                 check writing straight into the packed operand buffer (SURVEY 8f-2)
    cyclip.py    CyCLIPLoss drop-in (loss.py:813-905): CLIP term on the kernels, consistency terms through D x D
                 moment matrices (SURVEY 8f-4)
    graphed.py   CUDA-graph capture of the loss forward + backward (launch-bound small batches)
    pair_stats.py  CLIP-blind pair statistics on the Gram-tile kernel (helpers.py:221-285, SURVEY 8f-4)
    retrieval.py  retrieval ranks and R@K (open_clip get_clip_metrics) on the Gram-tile kernel, no N x N logits
    knn.py       kNN top-k neighbours and DINO's weighted kNN classifier on the Gram-tile kernel: per-strip top-k
                 lists in registers + a merge, no N_query x N_key score matrix
    geometry.py  embedding geometry (Wang & Isola uniformity and alignment, anisotropy, pairwise-cosine histograms)
                 on the Gram-tile kernel, no N x N matrix
    siglip.py    SigLipLoss drop-in (open_clip SigLipLoss): sigmoid loss and its logit gradient in one tile pass,
                 backward = the two gradient GEMMs, no B x B logit matrix
    distill.py   DistillClipLoss drop-in (open_clip DistillClipLoss): student and teacher row statistics in the
                 forward tile pass, one fp16 logit-gradient matrix + the two gradient GEMMs, no B x B logit matrix
    _cabi.py     ctypes binding of libdsoft.so (include/dsoft.h)
    _build.py    nvcc recipe for csrc/ (sm_100a only)
    csrc/        hand-written tcgen05 / TMEM / TMA kernels + the C ABI
"""
from . import _build, _cabi
from ._build import build
from .feature_store import DinoFeatureStore, DinoRows, lookup as dino_lookup, to_device_table
from .cyclip import CyCLIPLoss
from .graphed import make_graphed
from .pair_stats import pair_stats
from .retrieval import clip_metrics, retrieval_ranks
from .knn import knn_classify, knn_topk
from .geometry import embedding_geometry, image_text_geometry
from .siglip import SigLipLoss
from .distill import DistillClipLoss
from .loss import (
    ClipLossWithDINOEnhancements,
    CudaBackend,
    compute_student_tau,
    gather_features,
    install_into_open_clip,
    uninstall_from_open_clip,
)

__version__ = "0.1.0"
__all__ = [
    "ClipLossWithDINOEnhancements",
    "CudaBackend",
    "compute_student_tau",
    "gather_features",
    "install_into_open_clip",
    "uninstall_from_open_clip",
    "build",
    "DinoFeatureStore",
    "DinoRows",
    "to_device_table",
    "dino_lookup",
    "pair_stats",
    "retrieval_ranks",
    "clip_metrics",
    "knn_topk",
    "knn_classify",
    "embedding_geometry",
    "image_text_geometry",
    "CyCLIPLoss",
    "SigLipLoss",
    "DistillClipLoss",
    "make_graphed",
]
