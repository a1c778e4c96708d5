"""Image <-> text retrieval ranks and R@K on the Gram-tile kernel, without an N_img x N_txt logit matrix.

open_clip's `get_clip_metrics` (open_clip_train/train.py) builds the full fp32 logit matrix and argsorts it in both
directions: 4 N_img N_txt bytes, 40 GB for a 100k x 100k pool.  A rank is a count, so `dsoft_retrieval_ranks`
streams the score tiles s = I . T^T through TMEM and counts, per image and per caption, the non-positive scores
above the positive's:

    rank_img[i] = #{j : t(j) != i, s_ij > p_i},   p_i = max over the captions j of image i of s_ij
    rank_txt[j] = #{i : i != t(j), s_ij > s_t(j),j}

where t(j) is the image caption j belongs to (default t(j) = j).  Without ties this is exactly get_clip_metrics'
`preds`; ties count in the query's favour (strict >), where argsort breaks them arbitrarily.  Features are used as
given (no normalisation, as in get_clip_metrics); a positive logit_scale does not change any order and is ignored.

bf16 features are multiplied as they are; fp32 and fp16 features are split into bf16 (hi, lo) parts
(pair_stats._operands_ab), which reproduces their scores to ~1e-5 for unit-norm rows.  A rank can therefore differ
from the exact one only for a query with a non-positive score within that distance of its positive's.
Scratch is O(N_img + N_txt); the arithmetic runs on the GPU only.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _cabi
from .pair_stats import _operands_ab

_DIRECTIONS = ("image_to_text", "text_to_image")


def _check_args(image_features: torch.Tensor, text_features: torch.Tensor,
                text_image: Optional[torch.Tensor]) -> Tuple[int, int]:
    """Shape checks that need no device work."""
    if image_features.dim() != 2 or text_features.dim() != 2:
        raise ValueError("image_features and text_features must be [N, d] matrices")
    n_img, n_txt = int(image_features.shape[0]), int(text_features.shape[0])
    if image_features.shape[1] != text_features.shape[1]:
        raise ValueError(f"feature widths differ: {image_features.shape[1]} (images) and {text_features.shape[1]} "
                         "(texts)")
    if n_img == 0 or n_txt == 0:
        raise ValueError("empty image or text pool")
    if text_image is None:
        if n_img != n_txt:
            raise ValueError(f"{n_img} images and {n_txt} texts: pass text_image, the image index of every text")
    else:
        if text_image.shape != (n_txt,):
            raise ValueError(f"text_image must have one entry per text, shape ({n_txt},); got {tuple(text_image.shape)}")
        if text_image.dtype.is_floating_point or text_image.dtype.is_complex or text_image.dtype == torch.bool:
            raise ValueError("text_image must hold integer image indices")
    return n_img, n_txt


def _check_map(text_image: torch.Tensor, n_img: int) -> None:
    """Range and coverage of the caption -> image map: one host synchronisation."""
    t = text_image.to(torch.int64)
    lo, hi = t.min(), t.max()
    covered = torch.zeros(n_img, dtype=torch.bool, device=t.device)
    covered[t.clamp(0, n_img - 1)] = True
    lo, hi, missing = torch.stack([lo, hi, (~covered).sum()]).tolist()
    if lo < 0 or hi >= n_img:
        raise ValueError(f"text_image entries must lie in [0, {n_img}); found {lo if lo < 0 else hi}")
    if missing:
        raise ValueError(f"{missing} image(s) have no text in text_image")


def _device(*ts: torch.Tensor) -> torch.device:
    for t in ts:
        if t is not None and t.device.type == "cuda":
            return t.device
    if not torch.cuda.is_available():
        raise RuntimeError("retrieval ranks (B200 build) need a CUDA sm_100 device; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def retrieval_ranks(image_features: torch.Tensor, text_features: torch.Tensor,
                    text_image: Optional[torch.Tensor] = None, check: bool = True
                    ) -> Tuple[torch.Tensor, torch.Tensor]:
    """(rank_img int64 [N_img], rank_txt int64 [N_txt]) on the device: 0-based position of the first positive.

    text_image: the image index of every text (int tensor [N_txt]); None means text j belongs to image j.  CPU tensors
    are copied to the current CUDA device.  check=False skips the map's range / coverage check, the only host
    synchronisation, so that the call can be captured in a CUDA graph; the caller then guarantees a valid map."""
    n_img, n_txt = _check_args(image_features, text_features, text_image)
    if check and text_image is not None:
        _check_map(text_image, n_img)
    dev = _device(image_features, text_features, text_image)
    if torch.cuda.current_device() != dev.index:
        torch.cuda.set_device(dev)
    a, b, k = _operands_ab(image_features.to(dev), text_features.to(dev))
    tmap = None if text_image is None else text_image.to(device=dev, dtype=torch.int32).contiguous()
    lib = _cabi.lib()
    scratch = torch.empty(int(lib.dsoft_retrieval_scratch_bytes(n_img, n_txt)), dtype=torch.uint8, device=dev)
    rank_img = torch.empty(n_img, dtype=torch.int32, device=dev)
    rank_txt = torch.empty(n_txt, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    _cabi.check(lib.dsoft_retrieval_ranks(a.data_ptr(), b.data_ptr(), k, n_img, n_txt,
                                          None if tmap is None else tmap.data_ptr(), rank_img.data_ptr(),
                                          rank_txt.data_ptr(), scratch.data_ptr(), stream),
                "dsoft_retrieval_ranks")
    return rank_img.to(torch.int64), rank_txt.to(torch.int64)


def metrics_from_ranks(rank_img: torch.Tensor, rank_txt: torch.Tensor, ks: Sequence[int] = (1, 5, 10)
                       ) -> Dict[str, float]:
    """get_clip_metrics' reduction of the 0-based ranks, bit for bit: mean + 1, floor(numpy median) + 1 (the mean of
    the two middle values for even N, unlike torch.median), mean(rank < k).  One device -> host copy."""
    parts = []
    for r in (rank_img, rank_txt):
        r = r.to(torch.int64)
        n = r.numel()
        srt = r.sort().values
        parts.append(torch.stack([r.sum(), srt[(n - 1) // 2], srt[n // 2]] + [(r < k).sum() for k in ks]))
    vals = torch.stack(parts).tolist()  # exact integers
    out: Dict[str, float] = {}
    for name, r, v in zip(_DIRECTIONS, (rank_img, rank_txt), vals):
        n = r.numel()
        # integer sums below 2^53 are exact in float64, so one division reproduces numpy's float64 mean
        out[f"{name}_mean_rank"] = v[0] / n + 1
        out[f"{name}_median_rank"] = float((v[1] + v[2]) // 2) + 1  # floor of the (exact) middle mean
        for k, c in zip(ks, v[3:]):
            out[f"{name}_R@{k}"] = c / n
    return out


def clip_metrics(image_features: torch.Tensor, text_features: torch.Tensor, logit_scale=None,
                 text_image: Optional[torch.Tensor] = None, ks: Sequence[int] = (1, 5, 10)) -> Dict[str, float]:
    """open_clip get_clip_metrics on the GPU kernel: {image_to_text,text_to_image}_{mean_rank,median_rank,R@k} as
    Python floats.  logit_scale is accepted for signature parity and ignored (a positive scale keeps every order)."""
    del logit_scale
    rank_img, rank_txt = retrieval_ranks(image_features, text_features, text_image)
    return metrics_from_ranks(rank_img, rank_txt, ks)
