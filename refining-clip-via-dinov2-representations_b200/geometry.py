"""Embedding geometry on the Gram-tile kernel: uniformity, anisotropy, alignment and pairwise-cosine histograms
without an N x N matrix.

Wang & Isola (2020) measure uniformity as `torch.pdist(x).pow(2).mul(-t).exp().mean().log()`: N(N-1)/2 fp32 distances
and one more copy of that size per element-wise step (50 GB each at Flickr30k's 158 915 captions).  Here
`dsoft_geometry` streams the Gram tiles of the pool through TMEM and reduces each pair to one exponential and one
histogram count.  Work O(N^2 d) on the tensor cores, memory O(N d).

    embedding_geometry(features, t=2.0, bins=0, range=(-1.0, 1.0))
      uniformity = log( 2 / (N (N-1)) sum_{i<j} exp(2 t (cos_ij - 1)) )   (= uniform_loss: |x^_i - x^_j|^2 = 2 - 2 cos)
      anisotropy = mean_{i != j} cos_ij   (Ethayarajh 2019), in closed form (|sum_i x^_i|^2 - sum_i |x^_i|^2) / (N (N-1))
                   in fp64: O(N d), no tile pass
      hist / below / above (bins > 0): the cosines of the pairs i < j, numpy.histogram's bins over [lo, hi) with the
                   last one closed, and the counts outside the range; sum(hist) + below + above == N (N-1) / 2

    image_text_geometry(image_features, text_features, text_image=None, bins=100, range=(-1.0, 1.0), alpha=2.0)
      pos_hist / neg_hist (+ _below / _above): the positives (t(j), j) and every other pair (i, j)
      alignment = mean_j (2 - 2 cos_t(j),j)^(alpha / 2)   (align_loss over the matched pairs)

cos_ij = <x_i, y_j> r_i r_j with r = 1 / max(||row||, 1e-12) in fp32, taken over the values the kernel multiplies, as
in knn.py: the operands are never normalised and re-rounded.  bf16 inputs are multiplied as they are; fp32 and fp16
inputs take the [hi | lo | hi] . [hi | hi | lo]^T split of pair_stats._operands_ab (~1e-5 for unit-norm rows).
text_image has retrieval.py's meaning and checks (t(j) = the image of text j; None: t(j) = j).  The results come back as
Python floats and CPU int64 tensors after one host synchronisation; CPU tensors are copied to the current CUDA device.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch

from . import _cabi
from .knn import _inv_norms
from .pair_stats import _operands_ab
from .retrieval import _check_args as _check_pairs, _check_map, _device

T_MAX = 20.0     # exp(2 t (cos - 1)) >= e^-80 stays a normal fp32 number
BINS_MAX = 256
_ANISO_ROWS = 1 << 16


def _check_features(name: str, x) -> None:
    if not isinstance(x, torch.Tensor) or x.dim() != 2:
        raise ValueError(f"{name} must be an [N, d] tensor")
    if not x.dtype.is_floating_point:
        raise ValueError(f"{name} must be floating point, got {x.dtype}")
    if x.shape[0] == 0 or x.shape[1] == 0:
        raise ValueError(f"{name} is empty")


def _check_hist(bins, rng) -> Tuple[float, float]:
    if isinstance(bins, bool) or not isinstance(bins, int) or not 0 <= bins <= BINS_MAX:
        raise ValueError(f"bins must be an int in [0, {BINS_MAX}], got {bins!r}")
    try:
        lo, hi = (float(v) for v in rng)
    except (TypeError, ValueError):
        raise ValueError(f"range must be a pair of numbers (lo, hi), got {rng!r}") from None
    if not (math.isfinite(lo) and math.isfinite(hi) and lo < hi):
        raise ValueError(f"range needs finite lo < hi, got ({lo}, {hi})")
    return lo, hi


def _prepare(x: torch.Tensor, y: torch.Tensor, dev: torch.device):
    """(row operand, column operand, K, row scales, column scales, d, lo offset of the split or None)."""
    xd = x.to(dev)
    a, b, width = _operands_ab(xd, xd if y is x else y.to(dev))
    split = not (x.dtype == y.dtype == torch.bfloat16)
    dp = width // 3 if split else width
    # split operands: a = [hi | lo | hi], b = [hi | hi | lo]
    ra = _inv_norms(a, dp, dp if split else None)
    rb = ra if y is x else _inv_norms(b, dp, 2 * dp if split else None)
    return a, b, width, ra, rb, dp, (dp if split else None)


def _anisotropy(a: torch.Tensor, dp: int, lo_at: Optional[int], r: torch.Tensor) -> torch.Tensor:
    """(|sum_i x^_i|^2 - sum_i |x^_i|^2) / (N (N-1)) in fp64 with x^_i = r_i x_i, x_i the row the kernel multiplies
    (hi + lo of a split operand); in row chunks, so that no fp64 copy of the whole set exists.  A device scalar."""
    n = a.shape[0]
    s = torch.zeros(dp, dtype=torch.float64, device=a.device)
    sq = torch.zeros((), dtype=torch.float64, device=a.device)
    for i0 in range(0, n, _ANISO_ROWS):
        x = a[i0:i0 + _ANISO_ROWS, :dp].double()
        if lo_at is not None:
            x += a[i0:i0 + _ANISO_ROWS, lo_at:lo_at + dp].double()
        x *= r[i0:i0 + _ANISO_ROWS, None].double()
        s += x.sum(0)
        sq += (x * x).sum()
    return (s @ s - sq) / (n * (n - 1))


def _run(a, b, width, n_a, n_b, ra, rb, tmap, t, alpha, lo, hi, bins, dev, want_pos_cos=False):
    """dsoft_geometry: (sums fp64 [2], hist int64 [.., bins + 2], pos_cos) on the device, no synchronisation."""
    lib = _cabi.lib()
    nbytes = int(lib.dsoft_geometry_scratch_bytes(n_a, n_b, bins))
    if nbytes == 0:
        raise _cabi.DsoftError(f"dsoft_geometry_scratch_bytes: {lib.dsoft_last_error().decode()}")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    sums = torch.empty(2, dtype=torch.float64, device=dev)
    hist = torch.empty((1 if n_b == 0 else 2, bins + 2), dtype=torch.int64, device=dev)
    pos_cos = torch.empty(n_b, dtype=torch.float32, device=dev) if want_pos_cos else None
    stream = torch.cuda.current_stream(dev).cuda_stream
    _cabi.check(lib.dsoft_geometry(a.data_ptr(), None if b is a else b.data_ptr(), width, n_a, n_b, ra.data_ptr(),
                                   None if rb is None else rb.data_ptr(), None if tmap is None else tmap.data_ptr(),
                                   float(t), float(alpha), lo, hi, bins, sums.data_ptr(),
                                   hist.data_ptr() if bins else None,
                                   None if pos_cos is None else pos_cos.data_ptr(), scratch.data_ptr(), stream),
                "dsoft_geometry")
    return sums, hist, pos_cos


def _to_host(*parts: torch.Tensor):
    """One device -> host copy of fp64 and int64 tensors (fp64 travels as its bits)."""
    flat = [p.reshape(-1) for p in parts]
    host = torch.cat([p.view(torch.int64) if p.dtype == torch.float64 else p for p in flat]).cpu()
    out, k = [], 0
    for p in flat:
        h = host[k:k + p.numel()]
        out.append(h.view(torch.float64) if p.dtype == torch.float64 else h)
        k += p.numel()
    return out


def embedding_geometry(features: torch.Tensor, t: float = 2.0, bins: int = 0,
                       range: Tuple[float, float] = (-1.0, 1.0)) -> Dict[str, object]:
    """{"uniformity", "anisotropy"} as Python floats and, for bins > 0, {"hist": CPU int64 [bins], "below", "above"}
    over the N (N-1) / 2 pairs i < j of the rows of `features` [N, d], N >= 2 (see the module doc)."""
    _check_features("features", features)
    n = int(features.shape[0])
    if n < 2:
        raise ValueError(f"features needs at least 2 rows, got {n}")
    if isinstance(t, bool) or not isinstance(t, (int, float)) or not 0.0 < t <= T_MAX:
        raise ValueError(f"t must lie in (0, {T_MAX}], got {t!r}")
    lo, hi = _check_hist(bins, range)
    dev = _device(features)
    if torch.cuda.current_device() != dev.index:
        torch.cuda.set_device(dev)
    a, b, width, ra, _, dp, lo_at = _prepare(features, features, dev)
    sums, hist, _ = _run(a, b, width, n, 0, ra, None, None, t, 1.0, lo, hi, bins, dev)
    aniso = _anisotropy(a, dp, lo_at, ra)
    sums_h, aniso_h, hist_h = _to_host(sums, aniso, hist)
    pairs = n * (n - 1) // 2
    out: Dict[str, object] = {"uniformity": math.log(float(sums_h[0]) / pairs), "anisotropy": float(aniso_h[0])}
    if bins:
        out["hist"], out["below"], out["above"] = hist_h[:bins].clone(), int(hist_h[bins]), int(hist_h[bins + 1])
    return out


def image_text_geometry(image_features: torch.Tensor, text_features: torch.Tensor,
                        text_image: Optional[torch.Tensor] = None, bins: int = 100,
                        range: Tuple[float, float] = (-1.0, 1.0), alpha: float = 2.0) -> Dict[str, object]:
    """{"alignment": float} and, for bins > 0, the histograms of the positive and the negative pairs as CPU int64
    tensors [bins] with their out-of-range counts: {"pos_hist", "pos_below", "pos_above", "neg_hist", "neg_below",
    "neg_above"}.  Totals: N_txt positives and N_img N_txt - N_txt negatives (see the module doc)."""
    _check_features("image_features", image_features)
    _check_features("text_features", text_features)
    n_img, n_txt = _check_pairs(image_features, text_features, text_image)
    if isinstance(alpha, bool) or not isinstance(alpha, (int, float)) or not (0.0 < alpha < math.inf):
        raise ValueError(f"alpha must be a finite number > 0, got {alpha!r}")
    lo, hi = _check_hist(bins, range)
    if text_image is not None:
        _check_map(text_image, n_img)
    dev = _device(image_features, text_features, text_image)
    if torch.cuda.current_device() != dev.index:
        torch.cuda.set_device(dev)
    a, b, width, ra, rb, _, _ = _prepare(image_features, text_features, dev)
    tmap = None if text_image is None else text_image.to(device=dev, dtype=torch.int32).contiguous()
    sums, hist, _ = _run(a, b, width, n_img, n_txt, ra, rb, tmap, 0.0, alpha, lo, hi, bins, dev)
    sums_h, hist_h = _to_host(sums, hist)
    out: Dict[str, object] = {"alignment": float(sums_h[1]) / n_txt}
    if bins:
        hist_h = hist_h.view(2, bins + 2)
        for k, name in enumerate(("pos", "neg")):
            out[f"{name}_hist"] = hist_h[k, :bins].clone()
            out[f"{name}_below"], out[f"{name}_above"] = int(hist_h[k, bins]), int(hist_h[k, bins + 1])
    return out
