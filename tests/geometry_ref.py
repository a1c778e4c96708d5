"""Written-down restatement of the embedding-geometry measures in fp64: the statement geometry.py is checked against.

    x^_i        = x_i / max(||x_i||, 1e-12)                       (F.normalize)
    cos_ij      = <x^_i, y^_j>
    uniformity  = log( 2 / (N (N-1)) sum_{i<j} exp(2 t (cos_ij - 1)) )       Wang & Isola (2020), uniform_loss
    anisotropy  = mean_{i != j} cos_ij                                        Ethayarajh (2019)
    alignment   = mean_j max(2 - 2 cos_t(j),j, 0)^(alpha / 2)                 Wang & Isola (2020), align_loss
    histogram   bin = floor((cos - lo) bins / (hi - lo)), cos == hi in the last bin, cos < lo "below", cos > hi "above"
                (numpy.histogram's bins, plus the two counts it drops)

The reference's eval_geometry.py is not available, so t, alpha and the binning are the published definitions, not a
copy of its choices.  Row blocks keep the memory at O(block * N); on a GPU tensor the blocks run there."""
from __future__ import annotations

import builtins
import math
from typing import Dict, Optional, Tuple

import torch


def unit(x: torch.Tensor) -> torch.Tensor:
    x = x.double()
    return x / x.norm(dim=1, keepdim=True).clamp_min(1e-12)


def bin_index(c: torch.Tensor, bins: int, lo: float, hi: float) -> torch.Tensor:
    """Slot of each cosine in [bins + 2]: the bins, then below (bins) and above (bins + 1)."""
    idx = torch.floor((c - lo) * (bins / (hi - lo))).to(torch.int64).clamp(0, bins - 1)
    idx = torch.where(c < lo, torch.full_like(idx, bins), idx)
    return torch.where(c > hi, torch.full_like(idx, bins + 1), idx)


def near_edge(c: torch.Tensor, bins: int, lo: float, hi: float, eps: float) -> torch.Tensor:
    """[bins + 1]: how many cosines lie within eps of each bin edge lo + k (hi - lo) / bins."""
    w = (hi - lo) / bins
    k = torch.round((c - lo) / w)
    near = ((c - (lo + k * w)).abs() <= eps) & (k >= 0) & (k <= bins)
    return torch.bincount(k[near].to(torch.int64), minlength=bins + 1)


class Acc:
    """Sums over blocks of cosines: exp terms, histogram, edge counts."""

    def __init__(self, t, bins, lo, hi, eps, dev):
        self.t, self.bins, self.lo, self.hi, self.eps = t, bins, lo, hi, eps
        self.esum = torch.zeros((), dtype=torch.float64, device=dev)
        self.hist = torch.zeros(bins + 2, dtype=torch.int64, device=dev)
        self.near = torch.zeros(bins + 1, dtype=torch.int64, device=dev)

    def add(self, c: torch.Tensor) -> None:
        if self.t:
            self.esum += torch.exp(2.0 * self.t * (c - 1.0)).sum()
        if self.bins:
            self.hist += torch.bincount(bin_index(c, self.bins, self.lo, self.hi), minlength=self.bins + 2)
            self.near += near_edge(c, self.bins, self.lo, self.hi, self.eps)


def embedding_geometry_ref(x: torch.Tensor, t: float = 2.0, bins: int = 0, range: Tuple[float, float] = (-1.0, 1.0),
                           eps: float = 0.0, block: int = 2048) -> Dict[str, object]:
    """{"uniformity", "anisotropy"} and, for bins > 0, "hist" [bins + 2] (below, above last) and "near" [bins + 1]: the
    pairs within eps of each edge.  Tensors stay on x's device."""
    xn = unit(x)
    n = xn.shape[0]
    acc = Acc(t, bins, float(range[0]), float(range[1]), eps, xn.device)
    for i0 in builtins.range(0, n, block):
        c = xn[i0:i0 + block] @ xn[i0:].t()                     # rows i0.., columns i0..
        rows = torch.arange(c.shape[0], device=xn.device)[:, None]
        cols = torch.arange(c.shape[1], device=xn.device)[None, :]
        acc.add(c[cols > rows])                                 # pairs i < j
    pairs = n * (n - 1) // 2
    s = xn.sum(0)
    out = {"uniformity": math.log(float(acc.esum) / pairs) if t else None,
           "anisotropy": float((s @ s - (xn * xn).sum()) / (n * (n - 1))), "pairs": pairs}
    if bins:
        out["hist"], out["near"] = acc.hist, acc.near
    return out


def image_text_geometry_ref(img: torch.Tensor, txt: torch.Tensor, text_image: Optional[torch.Tensor] = None,
                            bins: int = 100, range: Tuple[float, float] = (-1.0, 1.0), alpha: float = 2.0,
                            eps: float = 0.0, block: int = 2048) -> Dict[str, object]:
    """{"alignment", "pos_cos"} and, for bins > 0, "pos_hist" / "neg_hist" [bins + 2] with "pos_near" / "neg_near"."""
    a, b = unit(img), unit(txt)
    n_img, n_txt = a.shape[0], b.shape[0]
    tmap = torch.arange(n_txt, device=a.device) if text_image is None else text_image.to(a.device, torch.int64)
    pos_cos = (a[tmap] * b).sum(1)
    lo, hi = float(range[0]), float(range[1])
    pos = Acc(0.0, bins, lo, hi, eps, a.device)
    neg = Acc(0.0, bins, lo, hi, eps, a.device)
    if bins:
        pos.add(pos_cos)
        for j0 in builtins.range(0, n_txt, block):
            c = a @ b[j0:j0 + block].t()                         # [n_img, block]
            positive = torch.zeros_like(c, dtype=torch.bool)
            cols = torch.arange(c.shape[1], device=a.device)
            positive[tmap[j0:j0 + block], cols] = True
            neg.add(c[~positive])
    out = {"alignment": float(alignment_ref(pos_cos, alpha)), "pos_cos": pos_cos}
    if bins:
        out.update(pos_hist=pos.hist, pos_near=pos.near, neg_hist=neg.hist, neg_near=neg.near)
    return out


def alignment_ref(pos_cos: torch.Tensor, alpha: float) -> torch.Tensor:
    return (2.0 - 2.0 * pos_cos.double()).clamp_min(0.0).pow(alpha / 2.0).mean()


def wang_isola_uniformity(x: torch.Tensor, t: float = 2.0) -> float:
    """Wang & Isola's uniform_loss as written (on F.normalize'd rows), in the dtype of x."""
    x = torch.nn.functional.normalize(x, dim=-1)
    return float(torch.pdist(x, p=2).pow(2).mul(-t).exp().mean().log())


def wang_isola_alignment(x: torch.Tensor, y: torch.Tensor, alpha: float = 2.0) -> float:
    """Wang & Isola's align_loss as written, on F.normalize'd matched rows."""
    x, y = torch.nn.functional.normalize(x, dim=-1), torch.nn.functional.normalize(y, dim=-1)
    return float((x - y).norm(p=2, dim=1).pow(alpha).mean())

