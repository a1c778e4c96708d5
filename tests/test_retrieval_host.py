"""Retrieval ranks (retrieval.py, dsoft_retrieval_ranks) on the CPU: the rank -> metric reduction against
get_clip_metrics' numpy formulas, the bf16 operand split, argument validation and the C-ABI surface."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT


def numpy_metrics(preds_img, preds_txt, ks=(1, 5, 10)):
    """The reduction of open_clip get_clip_metrics (open_clip_train/train.py) applied to given 0-based ranks."""
    metrics = {}
    for name, preds in (("image_to_text", preds_img), ("text_to_image", preds_txt)):
        metrics[f"{name}_mean_rank"] = preds.mean() + 1
        metrics[f"{name}_median_rank"] = np.floor(np.median(preds)) + 1
        for k in ks:
            metrics[f"{name}_R@{k}"] = np.mean(preds < k)
    return metrics


@pytest.mark.parametrize("n", [1, 2, 3, 10, 11, 1000, 4133])
def test_metrics_match_numpy_formulas(pkg, n):
    from dinosoft_b200.retrieval import metrics_from_ranks

    g = torch.Generator().manual_seed(n)
    for spread in (2, 7, 5 * n):
        ri = torch.randint(0, spread, (n,), generator=g)
        rt = torch.randint(0, spread, (n + 3,), generator=g)
        got = metrics_from_ranks(ri, rt)
        want = numpy_metrics(ri.numpy(), rt.numpy())
        assert list(got) == list(want)
        for key in want:
            assert isinstance(got[key], float)
            assert got[key] == float(want[key]), (key, got[key], want[key])


def test_even_median_is_numpy_not_torch(pkg):
    """numpy averages the two middle values (then floor), torch.median takes the lower one."""
    from dinosoft_b200.retrieval import metrics_from_ranks

    r = torch.tensor([0, 0, 5, 9])
    got = metrics_from_ranks(r, torch.tensor([1, 4]), ks=(1,))
    assert got["image_to_text_median_rank"] == np.floor(np.median(r.numpy())) + 1 == 3.0
    assert got["text_to_image_median_rank"] == 3.0  # floor(2.5) + 1
    assert float(torch.median(r)) + 1 == 1.0


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("d", [500, 512, 13])
def test_operand_split(pkg, dtype, d):
    from dinosoft_b200.pair_stats import _operands_ab

    g = torch.Generator().manual_seed(d)
    x = torch.nn.functional.normalize(torch.randn(37, d, generator=g), dim=-1).to(dtype)
    y = torch.nn.functional.normalize(torch.randn(29, d, generator=g), dim=-1).to(dtype)
    a, b, k = _operands_ab(x, y)
    dp = d + (-d) % 8
    assert a.dtype == b.dtype == torch.bfloat16 and a.is_contiguous() and b.is_contiguous()
    assert k % 8 == 0 and a.shape == (37, k) and b.shape == (29, k)
    exact = x.double() @ y.double().t()
    got = a.double() @ b.double().t()
    if dtype == torch.bfloat16:
        assert k == dp
        assert torch.equal(got, exact)
    else:
        assert k == 3 * dp
        hi, lo = a[:, :dp].double(), a[:, dp:2 * dp].double()
        assert torch.equal(a[:, 2 * dp:], a[:, :dp]) and torch.equal(b[:, dp:2 * dp], b[:, :dp])
        assert torch.all(a[:, d:dp] == 0)
        if dtype == torch.float16:  # fp16 -> hi + lo is exact, only lo . lo is dropped
            assert torch.equal(hi[:, :d] + lo[:, :d], x.double())
        assert (got - exact).abs().max().item() < (4e-6 if dtype == torch.float16 else 1e-5)


def test_split_of_one_matrix_matches_pair_stats(pkg):
    from dinosoft_b200.pair_stats import _operands, _operands_ab

    z = torch.randn(20, 36)
    for got, want in zip(_operands(z), _operands_ab(z, z.clone())):
        assert torch.equal(torch.as_tensor(got), torch.as_tensor(want))


@pytest.mark.parametrize("case, msg", [
    ("width", "feature widths differ"),
    ("missing_map", "pass text_image"),
    ("map_range", "must lie in"),
    ("map_negative", "must lie in"),
    ("no_caption", "have no text"),
    ("map_shape", "one entry per text"),
    ("map_float", "integer image indices"),
    ("empty", "empty"),
])
def test_argument_validation(pkg, case, msg):
    img, txt, tm = torch.randn(4, 16), torch.randn(8, 16), torch.tensor([0, 1, 2, 3, 0, 1, 2, 3])
    if case == "width":
        txt = torch.randn(8, 24)
    elif case == "missing_map":
        tm = None
    elif case == "map_range":
        tm = torch.tensor([0, 1, 2, 4, 0, 1, 2, 3])
    elif case == "map_negative":
        tm = torch.tensor([0, 1, 2, -1, 0, 1, 2, 3])
    elif case == "no_caption":
        tm = torch.tensor([0, 1, 2, 2, 0, 1, 2, 0])
    elif case == "map_shape":
        tm = tm[:7]
    elif case == "map_float":
        tm = tm.float()
    elif case == "empty":
        img, txt, tm = img[:0], txt[:0], None
    with pytest.raises(ValueError, match=msg):
        pkg.retrieval_ranks(img, txt, tm)
    with pytest.raises(ValueError, match=msg):
        pkg.clip_metrics(img, txt, 100.0, text_image=tm)


def test_no_cpu_fallback(pkg):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.retrieval_ranks(torch.randn(4, 16), torch.randn(4, 16))


def header_text():
    return open(os.path.join(ROOT, "include", "dsoft.h")).read()


def test_symbols_in_header_and_prototypes(pkg):
    from dinosoft_b200 import _cabi

    h = header_text()
    for name in ("dsoft_retrieval_scratch_bytes", "dsoft_retrieval_ranks"):
        assert re.search(rf"\b{name}\s*\(", h), name
        assert name in _cabi.PROTOTYPES
    assert int(re.search(r"#define DSOFT_VERSION (\d+)", h).group(1)) >= 250


def test_c_abi_host_side(pkg):
    """Sizes and argument checks that return before any device work."""
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    assert lib.dsoft_version() >= 250
    assert lib.dsoft_retrieval_scratch_bytes(0, 5) == 0
    # thr + map padded to 256 columns, p padded to 64 rows, 4 bytes each: O(N_img + N_txt)
    assert lib.dsoft_retrieval_scratch_bytes(1, 1) == 4 * (2 * 256 + 64)
    assert lib.dsoft_retrieval_scratch_bytes(1000, 5000) == 4 * (2 * 5120 + 1024)
    assert lib.dsoft_retrieval_scratch_bytes(131072, 131072) == 4 * (3 * 131072)
    buf = (C.c_int32 * 64)()
    p = C.addressof(buf)
    for args in [(None, p, 8, 4, 4, None, p, p, p, None),   # null operand
                 (p, p, 12, 4, 4, None, p, p, p, None),     # k not a multiple of 8
                 (p, p, 8, 0, 4, None, p, p, p, None),      # empty pool
                 (p, p, 8, 4, 5, None, p, p, p, None)]:     # no map for a non-square pool
        assert lib.dsoft_retrieval_ranks(*args) == -1
        assert lib.dsoft_last_error()
