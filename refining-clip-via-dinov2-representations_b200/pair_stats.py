"""CLIP-blind pair statistics on the B200 Gram-tile kernel (SURVEY 8f-4).

Mirror of the reference's `_pair_stats(clip_Z, dino_Z, thresholds)` (src/open_clip_train/helpers.py:221-285): same
arguments, same result dictionary (`total_pairs`, `thresholds`, `results[...]` with `count`, `percent`,
`clip_high_count`, `relative_percent`, and `top_pairs`).  The reference materialises two N x N fp32 cosine
matrices, the N(N-1)/2-element upper-triangle index tensors and one boolean mask per threshold; here
`dsoft_pair_stats` streams the upper block triangle of both Gram matrices through TMEM, counts in registers and only
writes the candidate pairs whose gap is large enough to be among the top `topk`.

fp32 inputs are split into bf16 (hi, lo) parts and multiplied as [hi | lo | hi] . [hi | hi | lo]^T: three bf16 tensor-
core products whose fp32 sum reproduces the fp32 cosine to ~1e-5, so a count can only differ from the reference's for
a pair that sits within that distance of a threshold.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Sequence, Tuple

import torch

from . import _cabi

_CAND_CAP = 1 << 20


def _operands(z: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, int]:
    """(row operand, column operand, K) as contiguous bf16 matrices whose product is z z^T."""
    return _operands_ab(z, z)


def _operands_ab(x: torch.Tensor, y: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, int]:
    """(row operand, column operand, K) as contiguous bf16 matrices whose product is x y^T.

    Two bf16 inputs are used as they are (widths zero-padded to a multiple of 8).  Anything else (fp32, and fp16,
    which bf16 does not hold exactly) is split into bf16 (hi, lo) and multiplied as [hi | lo | hi] . [hi | hi | lo]^T.
    """
    if x.dim() != 2 or y.dim() != 2:
        raise ValueError("expected [N, d] matrices")
    if x.shape[1] != y.shape[1]:
        raise ValueError(f"feature widths differ ({x.shape[1]} and {y.shape[1]})")
    d = x.shape[1]
    pad = (-d) % 8

    def padded(t):
        return torch.nn.functional.pad(t, (0, pad)) if pad else t

    if x.dtype == torch.bfloat16 and y.dtype == torch.bfloat16:
        a = padded(x).contiguous()
        return a, (a if y is x else padded(y).contiguous()), d + pad

    def split(t):
        t32 = t.float()
        hi = t32.to(torch.bfloat16)
        return padded(hi), padded((t32 - hi.float()).to(torch.bfloat16))

    xh, xl = split(x)
    yh, yl = (xh, xl) if y is x else split(y)
    a = torch.cat([xh, xl, xh], dim=1).contiguous()
    b = torch.cat([yh, yh, yl], dim=1).contiguous()
    return a, b, 3 * (d + pad)


def pair_stats(clip_Z: torch.Tensor, dino_Z: torch.Tensor, thresholds: Sequence[Tuple[float, float]],
               topk: int = 200) -> dict:
    """Same contract as helpers.py:221-285 (rows of both matrices L2-normalised, same row order)."""
    if clip_Z.device.type != "cuda" or dino_Z.device != clip_Z.device:
        raise RuntimeError("pair_stats (B200 build) needs CUDA tensors on one sm_100 device; there is no CPU fallback")
    if clip_Z.shape[0] != dino_Z.shape[0]:
        raise ValueError("clip_Z and dino_Z must have the same number of rows")
    thresholds = list(thresholds)
    if len(thresholds) > 8:
        raise ValueError("at most 8 threshold pairs per call")
    n = int(clip_Z.shape[0])
    total_pairs = n * (n - 1) // 2
    out = {"total_pairs": total_pairs, "results": {}, "thresholds": thresholds}
    if n < 2:
        for cmin, dmax in thresholds:
            out["results"][f"clip≥{cmin}_dino≤{dmax}"] = {"count": 0, "percent": 0.0, "clip_high_count": 0,
                                                          "relative_percent": 0.0}
        out["top_pairs"] = []
        return out
    lib = _cabi.lib()
    dev = clip_Z.device
    if torch.cuda.current_device() != dev.index:
        torch.cuda.set_device(dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    ca, cb, kc = _operands(clip_Z)
    da, db, kd = _operands(dino_Z)
    nt = len(thresholds)
    cmin = (C.c_float * max(nt, 1))(*[float(t[0]) for t in thresholds])
    dmax = (C.c_float * max(nt, 1))(*[float(t[1]) for t in thresholds])
    counts = torch.zeros(16, dtype=torch.int64, device=dev)
    cand = torch.empty((_CAND_CAP, 4), dtype=torch.float32, device=dev)
    ccount = torch.zeros(1, dtype=torch.int32, device=dev)
    want = min(int(topk), total_pairs)

    def run(floor: float, with_counts: bool, cap: int) -> int:
        ccount.zero_()
        _cabi.check(
            lib.dsoft_pair_stats(ca.data_ptr(), cb.data_ptr(), kc, da.data_ptr(), db.data_ptr(), kd, n, cmin, dmax,
                                 nt if with_counts else 0, counts.data_ptr() if with_counts else None, float(floor),
                                 cand.data_ptr() if cap else None, cap, ccount.data_ptr(), stream),
            "dsoft_pair_stats")
        return int(ccount.item()) & 0xFFFFFFFF

    # the gap floor is searched from above: a pass costs about a millisecond at N = 32768
    floor, step = 0.5, 0.25
    got = run(floor, True, _CAND_CAP if want else 0)
    while want and got < want and floor > -2.5:
        floor -= step
        got = run(floor, False, _CAND_CAP)
    while want and got > _CAND_CAP:  # too many above the floor to store: bisect upwards
        step *= 0.5
        floor += step
        got = run(floor, False, _CAND_CAP)
        if got < want:
            floor -= step
            step *= 0.5
            got = run(floor, False, _CAND_CAP)
            if got > _CAND_CAP and step < 1e-4:
                raise RuntimeError("pair_stats: more than 2^20 pairs tie at the gap of the top-k boundary")
    cnt = counts.cpu().tolist()
    for k, (cmin_k, dmax_k) in enumerate(thresholds):
        clip_high, blind = int(cnt[2 * k]), int(cnt[2 * k + 1])
        out["results"][f"clip≥{cmin_k}_dino≤{dmax_k}"] = {
            "count": blind,
            "percent": 100.0 * blind / (total_pairs or 1),
            "clip_high_count": clip_high,
            "relative_percent": 100.0 * blind / (clip_high or 1),
        }
    top: List[dict] = []
    if want:
        c = cand[:min(got, _CAND_CAP)]
        ij = c[:, :2].contiguous().view(torch.int32)
        gap = c[:, 2] - c[:, 3]
        # largest gaps first; ties in row-major pair order (the order of the reference's upper-triangle vector)
        key = ij[:, 0].to(torch.int64) * n + ij[:, 1].to(torch.int64)
        order = torch.argsort(key)
        order = order[torch.argsort(gap[order], descending=True, stable=True)][:want]
        sel, sij = c[order].cpu(), ij[order].cpu()
        top = [{"i": int(sij[r, 0]), "j": int(sij[r, 1]), "clip_sim": float(sel[r, 2]), "dino_sim": float(sel[r, 3]),
                "gap": float(sel[r, 2] - sel[r, 3])} for r in range(sel.shape[0])]
    out["top_pairs"] = top
    return out
