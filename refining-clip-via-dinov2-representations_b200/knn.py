"""kNN classification and top-k neighbours on the Gram-tile kernel, without an N_query x N_key similarity matrix.

DINO's `knn_classifier` (Caron et al. 2021, eval_knn.py) L2-normalises the features, builds `test_chunk @ train.T`
over the whole train set for each chunk of test queries, takes `topk(k)` and lets each neighbour vote for its class
with weight exp(s / T).  At ImageNet shape (50 000 x 1 281 167) the full fp32 score matrix would be 256 GB, and even
chunked the recipe writes, re-reads and row-sorts every score.  `dsoft_knn_topk` streams the score tiles through TMEM
instead and keeps, per query, the best keys of each column strip in registers; a merge kernel picks the top-k.  Work
O(N_q N_k d) on the tensor cores, output and scratch O(N_q k + N_k).

    knn_topk(queries, keys, k, normalize=False) -> (values fp32 [N_q, k], indices int64 [N_q, k])

Row i holds the k largest s_ij = <q_i, k_j> (normalize: divided by ||q_i|| ||k_j||) by decreasing value; equal values
come by increasing key index (stable and deterministic, where torch.topk leaves the order unspecified).
The operands are never normalised: 1/||k_j|| and 1/||q_i|| are fp32 scales applied to the fp32 product, computed from
the values the kernel multiplies (the bf16 operands, or hi + lo of split fp32 / fp16 inputs).  Normalising first and
rounding back to bf16 would move the scores by about 2^-9 relative.  bf16 inputs are multiplied as they are; fp32 and
fp16 inputs take the [hi | lo | hi] . [hi | hi | lo]^T split of pair_stats._operands_ab (~1e-5 for unit-norm rows).

    knn_classify(train_features, train_labels, test_features, test_labels, k=20, T=0.07, num_classes=None)

DINO's weighted vote: probs[i, c] = sum over the top-k neighbours n of query i with label c of exp(s_in / T), on
cosine scores; top-1 / top-5 accuracy in percent.  Classes of equal probability are ranked by class index (DINO's
`probs.sort` leaves them in arbitrary order).
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple, Union

import torch

from . import _cabi
from .pair_stats import _operands_ab
from .retrieval import _device

K_MAX = 64


def _check_args(queries: torch.Tensor, keys: torch.Tensor, k: int) -> Tuple[int, int]:
    """Shape and k checks that need no device work."""
    if not isinstance(queries, torch.Tensor) or not isinstance(keys, torch.Tensor):
        raise ValueError("queries and keys must be tensors")
    if queries.dim() != 2 or keys.dim() != 2:
        raise ValueError("queries and keys must be [N, d] matrices")
    if queries.shape[1] != keys.shape[1]:
        raise ValueError(f"feature widths differ: {queries.shape[1]} (queries) and {keys.shape[1]} (keys)")
    for name, t in (("queries", queries), ("keys", keys)):
        if not t.dtype.is_floating_point:
            raise ValueError(f"{name} must be floating point, got {t.dtype}")
    n_q, n_k = int(queries.shape[0]), int(keys.shape[0])
    if n_q == 0 or n_k == 0 or queries.shape[1] == 0:
        raise ValueError("empty query or key set")
    if isinstance(k, bool) or not isinstance(k, int):
        raise ValueError(f"k must be an int, got {k!r}")
    if not 1 <= k <= K_MAX:
        raise ValueError(f"k must lie in [1, {K_MAX}], got {k}")
    if k > n_k:
        raise ValueError(f"k = {k} exceeds the number of keys ({n_k})")
    return n_q, n_k


def _inv_norms(op: torch.Tensor, width: int, lo_at: Optional[int]) -> torch.Tensor:
    """1 / ||row|| in fp32 of the values the kernel multiplies: the bf16 row op[:, :width], plus the lo part at
    columns lo_at.. of a split operand.  A zero row gets 1e12 (F.normalize's eps): its scores stay 0."""
    x = op[:, :width].float()
    if lo_at is not None:
        x = x + op[:, lo_at:lo_at + width].float()
    return x.norm(dim=1).clamp_min(1e-12).reciprocal().contiguous()


def knn_topk(queries: torch.Tensor, keys: torch.Tensor, k: int, normalize: bool = False
             ) -> Tuple[torch.Tensor, torch.Tensor]:
    """(values fp32 [N_q, k], indices int64 [N_q, k]) on the device: the k best keys of every query (see module doc).
    CPU tensors are copied to the current CUDA device.  No host synchronisation (graph-capturable)."""
    n_q, n_k = _check_args(queries, keys, k)
    dev = _device(queries, keys)
    if torch.cuda.current_device() != dev.index:
        torch.cuda.set_device(dev)
    a, b, width = _operands_ab(queries.to(dev), keys.to(dev))
    qscale = kscale = None
    if normalize:
        split = not (queries.dtype == keys.dtype == torch.bfloat16)
        dp = width // 3 if split else width
        # split operands: a = [hi | lo | hi], b = [hi | hi | lo]
        qscale = _inv_norms(a, dp, dp if split else None)
        kscale = _inv_norms(b, dp, 2 * dp if split else None)
    lib = _cabi.lib()
    nbytes = int(lib.dsoft_knn_scratch_bytes(n_q, n_k, k))
    if nbytes == 0:
        raise _cabi.DsoftError(f"dsoft_knn_scratch_bytes: {lib.dsoft_last_error().decode()}")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    values = torch.empty((n_q, k), dtype=torch.float32, device=dev)
    indices = torch.empty((n_q, k), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    _cabi.check(lib.dsoft_knn_topk(a.data_ptr(), b.data_ptr(), width, n_q, n_k, k,
                                   None if kscale is None else kscale.data_ptr(),
                                   None if qscale is None else qscale.data_ptr(), values.data_ptr(),
                                   indices.data_ptr(), scratch.data_ptr(), stream),
                "dsoft_knn_topk")
    return values, indices.to(torch.int64)


def _check_labels(train_labels: torch.Tensor, test_labels: torch.Tensor, n_train: int, n_test: int,
                  num_classes: Optional[int]) -> int:
    """Shapes, dtypes and the label range [0, C): one host synchronisation.  Returns C."""
    for name, lab, n in (("train_labels", train_labels, n_train), ("test_labels", test_labels, n_test)):
        if not isinstance(lab, torch.Tensor) or lab.shape != (n,):
            shape = tuple(lab.shape) if isinstance(lab, torch.Tensor) else type(lab).__name__
            raise ValueError(f"{name} must have one entry per feature row, shape ({n},); got {shape}")
        if lab.dtype.is_floating_point or lab.dtype.is_complex or lab.dtype == torch.bool:
            raise ValueError(f"{name} must hold integer class indices, got {lab.dtype}")
    if num_classes is not None and (isinstance(num_classes, bool) or not isinstance(num_classes, int)
                                    or num_classes < 1):
        raise ValueError(f"num_classes must be a positive int, got {num_classes!r}")
    tr, te = train_labels.to(torch.int64), test_labels.to(device=train_labels.device, dtype=torch.int64)
    lo_tr, hi_tr, lo_te, hi_te = torch.stack([tr.min(), tr.max(), te.min(), te.max()]).tolist()
    c = num_classes if num_classes is not None else max(hi_tr, hi_te) + 1
    for name, mn, mx in (("train_labels", lo_tr, hi_tr), ("test_labels", lo_te, hi_te)):
        if mn < 0 or mx >= c:
            raise ValueError(f"{name} entries must lie in [0, {c}); found {mn if mn < 0 else mx}")
    return int(c)


def knn_classify(train_features: torch.Tensor, train_labels: torch.Tensor, test_features: torch.Tensor,
                 test_labels: torch.Tensor, k: Union[int, Sequence[int]] = 20, T: float = 0.07,
                 num_classes: Optional[int] = None) -> Dict[str, float]:
    """DINO's weighted kNN classifier on the kernel: {"knn_top1@k": %, "knn_top5@k": %} for every k as Python floats.

    k may be a sequence: the top-k runs once at max(k) and each k uses the first k neighbours of every row.  Top-5
    counts the label among the first min(5, k) classes.  num_classes None: max label + 1."""
    ks = [k] if isinstance(k, int) and not isinstance(k, bool) else list(k)
    if not ks:
        raise ValueError("k must be an int or a non-empty sequence of ints")
    kmax = max(ks) if all(isinstance(x, int) and not isinstance(x, bool) for x in ks) else None
    if kmax is None:
        raise ValueError(f"k must be an int or a sequence of ints, got {k!r}")
    for kk in ks:
        _check_args(test_features, train_features, kk)
    if not T > 0:
        raise ValueError(f"T must be > 0, got {T}")
    n_train, n_test = int(train_features.shape[0]), int(test_features.shape[0])
    c = _check_labels(train_labels, test_labels, n_train, n_test, num_classes)
    dev = _device(test_features, train_features)
    values, indices = knn_topk(test_features, train_features, kmax, normalize=True)
    train_lab = train_labels.to(device=dev, dtype=torch.int64)
    test_lab = test_labels.to(device=dev, dtype=torch.int64).view(-1, 1)
    neighbour_lab = train_lab[indices]                 # [N_q, kmax]
    weight = (values / T).exp()
    counts = []
    for kk in ks:
        probs = torch.zeros((n_test, c), dtype=torch.float32, device=dev)
        probs.scatter_add_(1, neighbour_lab[:, :kk], weight[:, :kk])
        order = torch.sort(probs, dim=1, descending=True, stable=True).indices  # ties: increasing class index
        correct = order[:, :min(5, kk)] == test_lab
        counts += [correct[:, 0].sum(), correct.sum()]
    counts = torch.stack(counts).tolist()
    out: Dict[str, float] = {}
    for n, kk in enumerate(ks):
        out[f"knn_top1@{kk}"] = counts[2 * n] * 100.0 / n_test
        out[f"knn_top5@{kk}"] = counts[2 * n + 1] * 100.0 / n_test
    return out
