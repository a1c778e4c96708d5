"""kNN top-k and classification (knn.py, dsoft_knn_topk) on the CPU: the fp64 restatement (tests/knn_ref.py) against
brute force and against DINO's recipe as written, argument validation and the C-ABI surface."""
import ctypes as C
import os
import re

import pytest
import torch

from conftest import ROOT
from knn_ref import dino_knn_classifier, knn_classify_ref, knn_topk_ref, stable_topk, vote


@pytest.mark.parametrize("normalize", [False, True])
@pytest.mark.parametrize("n_q, n_k, k", [(1, 1, 1), (7, 30, 5), (13, 64, 64), (5, 100, 20)])
def test_ref_topk_is_brute_force(normalize, n_q, n_k, k):
    g = torch.Generator().manual_seed(n_q * 1000 + n_k)
    if normalize:  # cosines of different vectors round differently: continuous features, no ties
        q, keys = torch.randn(n_q, 6, generator=g).double(), torch.randn(n_k, 6, generator=g).double()
    else:  # small integers: exact scores, many ties
        q = torch.randint(-3, 4, (n_q, 6), generator=g).double()
        keys = torch.randint(-3, 4, (n_k, 6), generator=g).double()
    vals, idx = knn_topk_ref(q, keys, k, normalize=normalize, block=4)
    for i in range(n_q):
        s = []
        for j in range(n_k):
            dot = float(q[i] @ keys[j])
            if normalize:
                dot /= max(float(q[i].norm()), 1e-12) * max(float(keys[j].norm()), 1e-12)
            s.append((dot, j))
        want = sorted(s, key=lambda p: (-p[0], p[1]))[:k]
        assert idx[i].tolist() == [j for _, j in want]
        assert vals[i].tolist() == pytest.approx([v for v, _ in want], abs=1e-12)


def test_ref_ties_by_index():
    s = torch.tensor([[1.0, 3.0, 3.0, 2.0, 3.0]])
    v, i = stable_topk(s, 4)
    assert i.tolist() == [[1, 2, 4, 3]] and v.tolist() == [[3.0, 3.0, 3.0, 2.0]]


def test_vote_orders_equal_classes_by_index():
    # k = 1: one class has the whole weight, every other class is 0 and they follow in index order
    vals, idx = torch.tensor([[0.5]]), torch.tensor([[0]])
    train = torch.tensor([7])
    for label in (7, 0, 3, 4):
        got = vote(vals, idx, train, torch.tensor([label]), 1, 0.07, 10)
        assert got == (int(label == 7), int(label == 7)), (label, got)  # min(5, k) = 1 class counts for top-5
    vals, idx = torch.tensor([[0.5, 0.5]]), torch.tensor([[0, 1]])
    train = torch.tensor([6, 2])  # equal weights: class 2 ranks first, then 6, then 0, 1, 3, ..
    assert vote(vals, idx, train, torch.tensor([2]), 2, 0.07, 10) == (1, 1)
    assert vote(vals, idx, train, torch.tensor([6]), 2, 0.07, 10) == (0, 1)
    assert vote(vals, idx, train, torch.tensor([0]), 2, 0.07, 10) == (0, 0)


def clustered(n_train, n_test, d, c, seed, spread=0.6):
    g = torch.Generator().manual_seed(seed)
    centres = torch.nn.functional.normalize(torch.randn(c, d, generator=g, dtype=torch.float64), dim=1)
    ytr = torch.randint(0, c, (n_train,), generator=g)
    yte = torch.randint(0, c, (n_test,), generator=g)
    xtr = centres[ytr] + spread * torch.randn(n_train, d, generator=g, dtype=torch.float64) / d ** 0.5
    xte = centres[yte] + spread * torch.randn(n_test, d, generator=g, dtype=torch.float64) / d ** 0.5
    return xtr, ytr, xte, yte


@pytest.mark.parametrize("k", [10, 20, 40])
def test_ref_matches_dino_recipe_without_ties(k):
    """On continuous features (no equal scores) and for queries with at least min(5, k) classes of nonzero weight,
    DINO's recipe has no order left to choose, and the stable restatement gives the same accuracies."""
    xtr, ytr, xte, yte = clustered(3000, 600, 32, 8, seed=k, spread=2.5)
    _, idx = knn_topk_ref(xte, xtr, k, normalize=True)
    distinct = torch.tensor([len(set(ytr[r].tolist())) for r in idx])
    keep = distinct >= min(5, k)  # elsewhere zero-weight classes reach the top 5 in DINO's arbitrary order
    assert int(keep.sum()) >= 100
    xte, yte = xte[keep], yte[keep]
    ntr = torch.nn.functional.normalize(xtr, dim=1)
    nte = torch.nn.functional.normalize(xte, dim=1)
    top1, top5 = dino_knn_classifier(ntr, ytr, nte, yte, k, 0.07, num_classes=8)
    ref = knn_classify_ref(xtr, ytr, xte, yte, k=k, T=0.07, num_classes=8)
    assert ref[f"knn_top1@{k}"] == top1 and ref[f"knn_top5@{k}"] == top5
    assert 20.0 < top1 < 100.0


def test_ref_sequence_k_is_prefix():
    xtr, ytr, xte, yte = clustered(500, 60, 16, 5, seed=3)
    both = knn_classify_ref(xtr, ytr, xte, yte, k=(3, 10))
    for k in (3, 10):
        one = knn_classify_ref(xtr, ytr, xte, yte, k=k)
        assert one == {key: v for key, v in both.items() if key.endswith(f"@{k}")}


@pytest.mark.parametrize("case, msg", [
    ("dims", r"\[N, d\] matrices"),
    ("width", "feature widths differ"),
    ("empty_q", "empty"),
    ("empty_k", "empty"),
    ("k0", r"k must lie in \[1, 64\]"),
    ("k65", r"k must lie in \[1, 64\]"),
    ("k_float", "k must be an int"),
    ("k_bool", "k must be an int"),
    ("k_gt_nk", "exceeds the number of keys"),
    ("int_features", "floating point"),
])
def test_topk_argument_validation(pkg, case, msg):
    q, keys, k = torch.randn(4, 16), torch.randn(8, 16), 3
    if case == "dims":
        q = q[0]
    elif case == "width":
        keys = torch.randn(8, 24)
    elif case == "empty_q":
        q = q[:0]
    elif case == "empty_k":
        keys = keys[:0]
    elif case == "k0":
        k = 0
    elif case == "k65":
        keys, k = torch.randn(100, 16), 65
    elif case == "k_float":
        k = 3.0
    elif case == "k_bool":
        k = True
    elif case == "k_gt_nk":
        k = 9
    elif case == "int_features":
        q = torch.ones(4, 16, dtype=torch.int32)
    with pytest.raises(ValueError, match=msg):
        pkg.knn_topk(q, keys, k)


@pytest.mark.parametrize("case, msg", [
    ("train_shape", "train_labels must have one entry"),
    ("test_shape", "test_labels must have one entry"),
    ("float_labels", "integer class indices"),
    ("bool_labels", "integer class indices"),
    ("negative", "must lie in"),
    ("too_large", "must lie in"),
    ("num_classes", "num_classes must be a positive int"),
    ("T", "T must be > 0"),
    ("k_empty", "non-empty sequence"),
    ("k_seq_bad", "k must be an int or a sequence of ints"),
    ("k_seq_range", r"k must lie in \[1, 64\]"),
    ("k_gt_ntrain", "exceeds the number of keys"),
])
def test_classify_argument_validation(pkg, case, msg):
    xtr, ytr, xte, yte = torch.randn(30, 16), torch.arange(30) % 4, torch.randn(6, 16), torch.arange(6) % 4
    kw = dict(k=5, T=0.07, num_classes=None)
    if case == "train_shape":
        ytr = ytr[:29]
    elif case == "test_shape":
        yte = yte.view(2, 3)
    elif case == "float_labels":
        ytr = ytr.float()
    elif case == "bool_labels":
        yte = yte > 1
    elif case == "negative":
        ytr = ytr.clone()
        ytr[3] = -1
    elif case == "too_large":
        kw["num_classes"] = 3
    elif case == "num_classes":
        kw["num_classes"] = 0
    elif case == "T":
        kw["T"] = 0.0
    elif case == "k_empty":
        kw["k"] = ()
    elif case == "k_seq_bad":
        kw["k"] = (5, 2.5)
    elif case == "k_seq_range":
        kw["k"] = (5, 70)
    elif case == "k_gt_ntrain":
        kw["k"] = 31
    with pytest.raises(ValueError, match=msg):
        pkg.knn_classify(xtr, ytr, xte, yte, **kw)


def test_no_cpu_fallback(pkg):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.knn_topk(torch.randn(4, 16), torch.randn(8, 16), 3)


def test_symbols_in_header_and_prototypes(pkg):
    from dinosoft_b200 import _cabi

    h = open(os.path.join(ROOT, "include", "dsoft.h")).read()
    for name in ("dsoft_knn_scratch_bytes", "dsoft_knn_topk"):
        m = re.search(rf"\b{name}\s*\(([^)]*)\)", h)
        assert m, name
        assert len(_cabi.PROTOTYPES[name][1]) == len([a for a in m.group(1).split(",") if a.strip()]), name


def test_c_abi_host_side(pkg):
    """Argument checks that return before any device work."""
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    for args in [(0, 5, 1), (5, 0, 1), (5, 5, 0), (5, 100, 65), (5, 4, 5)]:
        assert lib.dsoft_knn_scratch_bytes(*args) == 0, args
    buf = (C.c_int32 * 64)()
    p = C.addressof(buf)
    for args in [(None, p, 8, 4, 4, 1, None, None, p, p, p, None),    # null operand
                 (p, p, 8, 4, 4, 1, None, None, None, p, p, None),    # null values
                 (p, p, 12, 4, 4, 1, None, None, p, p, p, None),      # width not a multiple of 8
                 (p, p, 8, 0, 4, 1, None, None, p, p, p, None),       # no queries
                 (p, p, 8, 4, 4, 0, None, None, p, p, p, None),       # k = 0
                 (p, p, 8, 4, 100, 65, None, None, p, p, p, None),    # k > 64
                 (p, p, 8, 4, 4, 5, None, None, p, p, p, None),       # k > n_k
                 (p + 4, p, 8, 4, 4, 1, None, None, p, p, p, None)]:  # misaligned operand
        assert lib.dsoft_knn_topk(*args) == -1, args
        assert lib.dsoft_last_error()
