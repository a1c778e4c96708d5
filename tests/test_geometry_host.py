"""Embedding geometry (geometry.py, dsoft_geometry) on the CPU: the fp64 restatement (tests/geometry_ref.py) against
Wang & Isola's recipe as written, against brute force and against numpy / torch histograms; argument validation and
the C-ABI surface."""
import ctypes as C
import itertools
import math
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from geometry_ref import (bin_index, embedding_geometry_ref, image_text_geometry_ref, near_edge, unit,
                          wang_isola_alignment, wang_isola_uniformity)


@pytest.mark.parametrize("n, d, t", [(2, 3, 2.0), (5, 8, 1.0), (37, 16, 2.0), (100, 7, 0.5), (64, 32, 20.0)])
def test_uniformity_is_wang_isola(n, d, t):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(n + d), dtype=torch.float64)
    ref = embedding_geometry_ref(x, t=t, block=16)
    assert ref["uniformity"] == pytest.approx(wang_isola_uniformity(x, t), rel=1e-12, abs=1e-12)


@pytest.mark.parametrize("alpha", [0.5, 1.0, 2.0, 3.0])
def test_alignment_is_wang_isola(alpha):
    g = torch.Generator().manual_seed(7)
    img, txt = torch.randn(20, 12, generator=g, dtype=torch.float64), torch.randn(50, 12, generator=g,
                                                                                 dtype=torch.float64)
    tmap = torch.randint(0, 20, (50,), generator=g)
    ref = image_text_geometry_ref(img, txt, tmap, bins=0, alpha=alpha)
    assert ref["alignment"] == pytest.approx(wang_isola_alignment(img[tmap], txt, alpha), rel=1e-12)


@pytest.mark.parametrize("n, d", [(2, 4), (9, 5), (60, 16)])
def test_anisotropy_closed_form_is_brute_force(n, d):
    x = torch.randn(n, d, generator=torch.Generator().manual_seed(n), dtype=torch.float64) + 0.7
    xn = unit(x)
    brute = sum(float(xn[i] @ xn[j]) for i, j in itertools.permutations(range(n), 2)) / (n * (n - 1))
    assert embedding_geometry_ref(x, block=4)["anisotropy"] == pytest.approx(brute, rel=1e-12, abs=1e-15)


def test_histogram_matches_numpy_in_range():
    g = torch.Generator().manual_seed(3)
    c = torch.rand(20000, generator=g, dtype=torch.float64) * 2 - 1
    # values exactly on edges, the closed last edge and both range ends (dyadic: exact in every formula)
    c = torch.cat([c, torch.arange(-16, 17, dtype=torch.float64) / 16])
    for bins, lo, hi in [(32, -1.0, 1.0), (7, -1.0, 1.0), (100, -1.0, 1.0), (256, -1.0, 1.0), (8, -0.5, 1.0)]:
        inside = c[(c >= lo) & (c <= hi)]
        want, _ = np.histogram(inside.numpy(), bins=bins, range=(lo, hi))
        got = torch.bincount(bin_index(inside, bins, lo, hi), minlength=bins + 2)
        assert got[:bins].tolist() == want.tolist(), (bins, lo, hi)
        assert int(got[bins:].sum()) == 0


def test_histogram_counts_what_histc_drops():
    g = torch.Generator().manual_seed(4)
    c = torch.randn(10000, generator=g, dtype=torch.float64) * 0.6
    bins, lo, hi = 50, -0.9, 0.8
    got = torch.bincount(bin_index(c, bins, lo, hi), minlength=bins + 2)
    histc = torch.histc(c, bins=bins, min=lo, max=hi)
    assert got[:bins].tolist() == histc.to(torch.int64).tolist()
    assert int(got[bins]) == int((c < lo).sum()) > 0 and int(got[bins + 1]) == int((c > hi).sum()) > 0
    assert int(got.sum()) == c.numel() and int(histc.sum()) < c.numel()


def test_near_edge():
    c = torch.tensor([-1.0, -1.0 + 1e-7, -0.5 - 2e-7, 0.0, 0.1, 1.0, 1.0 + 5e-8], dtype=torch.float64)
    near = near_edge(c, 4, -1.0, 1.0, 1e-6)
    assert near.tolist() == [2, 1, 1, 0, 2]


def test_restatement_totals():
    g = torch.Generator().manual_seed(5)
    x = torch.randn(77, 6, generator=g)
    ref = embedding_geometry_ref(x, bins=10, range=(-0.5, 0.5), block=8)
    assert int(ref["hist"].sum()) == 77 * 76 // 2 and int(ref["hist"][10:].sum()) > 0
    img, txt = torch.randn(9, 6, generator=g), torch.randn(30, 6, generator=g)
    tmap = torch.arange(30) % 9
    r = image_text_geometry_ref(img, txt, tmap, bins=10, block=7)
    assert int(r["pos_hist"].sum()) == 30 and int(r["neg_hist"].sum()) == 9 * 30 - 30


@pytest.mark.parametrize("case, msg", [
    ("dims", r"\[N, d\] tensor"),
    ("int", "floating point"),
    ("empty", "empty"),
    ("one_row", "at least 2 rows"),
    ("t0", r"t must lie in \(0, 20"),
    ("t_big", r"t must lie in \(0, 20"),
    ("t_nan", r"t must lie in \(0, 20"),
    ("bins_neg", r"bins must be an int in \[0, 256\]"),
    ("bins_big", r"bins must be an int in \[0, 256\]"),
    ("bins_float", "bins must be an int"),
    ("range_order", "finite lo < hi"),
    ("range_inf", "finite lo < hi"),
    ("range_shape", "pair of numbers"),
])
def test_embedding_argument_validation(pkg, case, msg):
    x, kw = torch.randn(6, 16), {}
    if case == "dims":
        x = x[0]
    elif case == "int":
        x = torch.ones(6, 16, dtype=torch.int32)
    elif case == "empty":
        x = x[:, :0]
    elif case == "one_row":
        x = x[:1]
    elif case == "t0":
        kw["t"] = 0.0
    elif case == "t_big":
        kw["t"] = 20.5
    elif case == "t_nan":
        kw["t"] = math.nan
    elif case == "bins_neg":
        kw["bins"] = -1
    elif case == "bins_big":
        kw["bins"] = 257
    elif case == "bins_float":
        kw["bins"] = 10.0
    elif case == "range_order":
        kw.update(bins=10, range=(0.5, 0.5))
    elif case == "range_inf":
        kw.update(bins=10, range=(-math.inf, 1.0))
    elif case == "range_shape":
        kw.update(bins=10, range=(0.0, 1.0, 2.0))
    with pytest.raises(ValueError, match=msg):
        pkg.embedding_geometry(x, **kw)


@pytest.mark.parametrize("case, msg", [
    ("width", "feature widths differ"),
    ("empty_txt", "empty"),
    ("no_map", "pass text_image"),
    ("map_shape", "one entry per text"),
    ("map_float", "integer image indices"),
    ("map_range", r"must lie in \[0, 4\)"),
    ("map_cover", "have no text"),
    ("alpha", "alpha must be a finite number > 0"),
    ("alpha_inf", "alpha must be a finite number > 0"),
    ("bins", r"bins must be an int in \[0, 256\]"),
])
def test_image_text_argument_validation(pkg, case, msg):
    img, txt, tmap, kw = torch.randn(4, 16), torch.randn(8, 16), torch.arange(8) % 4, {}
    if case == "width":
        txt = torch.randn(8, 24)
    elif case == "empty_txt":
        txt = txt[:0]
    elif case == "no_map":
        tmap = None
    elif case == "map_shape":
        tmap = tmap[:7]
    elif case == "map_float":
        tmap = tmap.float()
    elif case == "map_range":
        tmap = tmap.clone()
        tmap[2] = 4
    elif case == "map_cover":
        tmap = torch.zeros(8, dtype=torch.int64)
    elif case == "alpha":
        kw["alpha"] = 0.0
    elif case == "alpha_inf":
        kw["alpha"] = math.inf
    elif case == "bins":
        kw["bins"] = 300
    with pytest.raises(ValueError, match=msg):
        pkg.image_text_geometry(img, txt, tmap, **kw)


def test_no_cpu_fallback(pkg):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.embedding_geometry(torch.randn(4, 16))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.image_text_geometry(torch.randn(4, 16), torch.randn(4, 16))


def test_exported(pkg):
    assert {"embedding_geometry", "image_text_geometry"} <= set(pkg.__all__)


def test_symbols_in_header_and_prototypes(pkg):
    from dinosoft_b200 import _cabi

    h = open(os.path.join(ROOT, "include", "dsoft.h")).read()
    for name in ("dsoft_geometry_scratch_bytes", "dsoft_geometry"):
        m = re.search(rf"\b{name}\s*\(([^)]*)\)", h)
        assert m, name
        assert len(_cabi.PROTOTYPES[name][1]) == len([a for a in m.group(1).split(",") if a.strip()]), name


def test_c_abi_host_side(pkg):
    """Argument checks that return DSOFT_EINVAL before any device work."""
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    for args in [(1, 0, 0), (0, 0, 10), (4, -1, 0), (0, 5, 0), (5, 0, -1), (5, 0, 257), (5, 5, 300)]:
        assert lib.dsoft_geometry_scratch_bytes(*args) == 0, args
    buf = (C.c_int64 * 64)()
    p = C.addressof(buf)
    ok = dict(a=p, b=None, width=8, n_a=4, n_b=0, ra=None, rb=None, tmap=None, t=2.0, alpha=2.0, lo=-1.0, hi=1.0,
              bins=10, sums=p, hist=p, pos=None, scratch=p, stream=None)
    bad = [dict(a=None), dict(sums=None), dict(scratch=None), dict(hist=None),    # null arguments
           dict(width=12), dict(width=0),                                        # width not a positive multiple of 8
           dict(n_a=1), dict(n_b=-2), dict(bins=257), dict(bins=-1),              # sizes
           dict(t=-1.0), dict(t=20.5), dict(t=math.nan),                          # t
           dict(lo=1.0, hi=1.0), dict(hi=math.inf),                               # range
           dict(tmap=p), dict(pos=p),                                             # one set has no positives
           dict(n_b=4, b=p, alpha=0.0), dict(n_b=4, b=p, alpha=math.nan),        # alpha
           dict(n_b=4),                                                          # two sets without b
           dict(n_b=5, b=p),                                                     # n_a != n_b without a map
           dict(a=p + 4)]                                                        # misaligned operand
    for change in bad:
        kw = {**ok, **change}
        assert lib.dsoft_geometry(*kw.values()) == -1, change
        assert lib.dsoft_last_error()
