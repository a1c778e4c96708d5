"""kNN top-k and classification (knn.py -> dsoft_knn_topk -> dsoft_fwd_kernel<MODE_TOPK / MODE_TOPK32> + the merge
kernel) against the fp64 restatement in tests/knn_ref.py, computed on the GPU in row blocks.

Rule, for query i with fp64 scores s (normalised when requested) and theta_i their k-th largest:
  * every j with s_ij > theta_i + eps is returned, and every returned j has s_ij >= theta_i - eps;
  * the indices are distinct and in range, and |value - s_ij| <= eps for each returned pair;
  * the values do not increase along the row, and equal values come in increasing index order.
eps = 2e-5 for split fp32 / fp16 inputs and 4e-6 for bf16 inputs, for unit-norm features; without normalize it is
scaled by ||q_i|| max_j ||k_j||.  Integer features make every score exact: the result then equals the fp64 stable
top-k, tie order included."""
import pytest
import torch

from knn_ref import knn_classify_ref, knn_topk_ref, scores

pytestmark = pytest.mark.gpu

EPS = {torch.float32: 2e-5, torch.float16: 2e-5, torch.bfloat16: 4e-6}


def check_topk(q, keys, vals, idx, k, normalize, eps, rows=None, block=256):
    """Apply the tolerance rule to the rows `rows` (default: all).  Returns the worst |value - s|."""
    dev = torch.device("cuda")
    qd, kd = q.to(dev), keys.to(dev)
    rows = torch.arange(q.shape[0], device=dev) if rows is None else rows.to(dev)
    n_k = keys.shape[0]
    assert vals.shape == idx.shape == (q.shape[0], k) and vals.dtype == torch.float32 and idx.dtype == torch.int64
    kmax = None if normalize else kd.float().norm(dim=1).max().double()
    worst = 0.0
    for r0 in range(0, rows.numel(), block):
        r = rows[r0:r0 + block]
        s = scores(qd[r], kd, normalize)
        e = torch.full((r.numel(), 1), eps, dtype=torch.float64, device=dev)
        if not normalize:
            e = e * qd[r].double().norm(dim=1, keepdim=True) * kmax
        theta = s.topk(k, dim=1).values[:, -1:]
        v, i = vals[r].to(dev).double(), idx[r].to(dev)
        assert bool(((i >= 0) & (i < n_k)).all())
        si = i.sort(dim=1).values
        assert bool((si[:, 1:] != si[:, :-1]).all()), "repeated index"
        got = torch.zeros_like(s, dtype=torch.bool).scatter_(1, i, True)
        assert not bool(((s > theta + e) & ~got).any()), "a clear neighbour is missing"
        sg = s.gather(1, i)
        assert bool((sg >= theta - e).all()), "a returned key is clearly outside the top-k"
        err = (v - sg).abs()
        assert bool((err <= e).all()), float(err.max())
        worst = max(worst, float(err.max()))
        assert bool((v[:, 1:] <= v[:, :-1]).all()), "values increase"
        tie = v[:, 1:] == v[:, :-1]
        assert bool((~tie | (i[:, 1:] > i[:, :-1])).all()), "equal values out of index order"
    return worst


def unit(n, d, seed, dtype, dev="cuda"):
    g = torch.Generator(device=dev).manual_seed(seed)
    return torch.nn.functional.normalize(torch.randn(n, d, device=dev, generator=g), dim=1).to(dtype)


# (n_q, n_k, k, d, dtype, normalize): every N_q of {1, 7, 255, 256, 257, 4133}, N_k of {k, 255, 257, 5000, 100003},
# k of {1, 5, 20, 64}, d of {8, 500, 512, 768, 1024} and each input dtype, with and without normalisation
CASES = [
    (1, 1, 1, 8, torch.bfloat16, False),
    (1, 64, 64, 500, torch.float32, True),
    (7, 5, 5, 512, torch.float16, True),
    (7, 255, 20, 768, torch.bfloat16, True),
    (255, 257, 64, 1024, torch.float32, False),
    (256, 255, 5, 512, torch.bfloat16, False),
    (257, 5000, 20, 8, torch.float32, True),
    (256, 5000, 64, 768, torch.float16, False),
    (4133, 5000, 20, 768, torch.bfloat16, True),
    (4133, 257, 1, 500, torch.float16, True),
    (255, 100003, 64, 768, torch.bfloat16, True),
    (257, 100003, 5, 1024, torch.float32, True),
    (1, 100003, 20, 512, torch.float32, False),
]


@pytest.mark.parametrize("n_q, n_k, k, d, dtype, normalize", CASES)
def test_topk_against_fp64(pkg, n_q, n_k, k, d, dtype, normalize):
    seed = n_q * 7 + n_k + k
    q, keys = unit(n_q, d, seed, dtype), unit(n_k, d, seed + 1, dtype)
    if not normalize:  # norms away from 1, so that the scales matter
        g = torch.Generator(device="cuda").manual_seed(seed + 2)
        q = (q.float() * (0.5 + 2 * torch.rand(n_q, 1, device="cuda", generator=g))).to(dtype)
        keys = (keys.float() * (0.5 + 2 * torch.rand(n_k, 1, device="cuda", generator=g))).to(dtype)
    else:  # and normalize has to undo them
        q = (q.float() * 3.0).to(dtype)
    vals, idx = pkg.knn_topk(q, keys, k, normalize=normalize)
    worst = check_topk(q, keys, vals, idx, k, normalize, EPS[dtype])
    print(f"[knn] {n_q}x{n_k} k={k} d={d} {dtype} normalize={normalize}: worst |value - fp64| {worst:.2e}")


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
@pytest.mark.parametrize("normalize", [False, True])
def test_noncontiguous_and_host_inputs(pkg, dtype, normalize):
    big_q, big_k = unit(300, 2 * 520, 11, dtype), unit(3000, 520, 12, dtype)
    q = big_q[:, ::2]            # strided columns
    keys = big_k.t().contiguous().t()  # column-major
    assert not q.is_contiguous() and not keys.is_contiguous()
    vals, idx = pkg.knn_topk(q, keys.cpu(), 20, normalize=normalize)  # a host tensor is copied to the device
    assert vals.is_cuda and idx.is_cuda
    check_topk(q, keys, vals, idx, 20, normalize, EPS[dtype])


@pytest.mark.parametrize("n_q, n_k, k, d, dtype", [
    (300, 2000, 64, 8, torch.bfloat16),
    (257, 5000, 20, 64, torch.float32),
    (33, 700, 5, 16, torch.float16),
    (5, 64, 64, 8, torch.bfloat16),
])
def test_exact_ties_integer_features(pkg, n_q, n_k, k, d, dtype):
    """Scores are small integers, exact in every arithmetic involved: the exact stable top-k, tie order included."""
    g = torch.Generator().manual_seed(n_k + k)
    q = torch.randint(-2, 3, (n_q, d), generator=g).to(dtype)
    keys = torch.randint(-2, 3, (n_k, d), generator=g).to(dtype)
    vals, idx = pkg.knn_topk(q.cuda(), keys.cuda(), k)
    want_v, want_i = knn_topk_ref(q.cuda(), keys.cuda(), k)
    assert torch.equal(idx, want_i)
    assert torch.equal(vals.double(), want_v)
    assert int((want_v[:, 1:] == want_v[:, :-1]).sum()) > n_q  # the case does exercise ties


@pytest.mark.parametrize("k", [5, 64])
def test_rising_scores_insert_every_key(pkg, k):
    """Scores rise along the key axis, so every key enters its strip's list: the insertion path on every score."""
    n_q, n_k, d = 300, 20000, 256
    q = unit(n_q, d, 21, torch.float32).abs()
    base = unit(1, d, 22, torch.float32).abs()
    g = torch.Generator(device="cuda").manual_seed(23)
    keys = base + 0.05 * torch.rand(n_k, d, device="cuda", generator=g)
    keys = keys * torch.linspace(0.5, 1.5, n_k, device="cuda")[:, None]
    vals, idx = pkg.knn_topk(q, keys, k)
    check_topk(q, keys, vals, idx, k, False, EPS[torch.float32])
    assert int(idx.min()) >= n_k // 2  # the late keys win


def test_class_sorted_keys(pkg):
    """Keys stored class by class (as an ImageNet train set is): a row's neighbours crowd into few strips."""
    c, per, d = 100, 200, 384
    centres = unit(c, d, 31, torch.float32)
    g = torch.Generator(device="cuda").manual_seed(32)
    keys = centres.repeat_interleave(per, 0) + 0.2 * torch.randn(c * per, d, device="cuda", generator=g) / d ** 0.5
    q = centres[torch.randint(0, c, (500,), device="cuda", generator=g)] + 0.2 * torch.randn(500, d, device="cuda",
                                                                                             generator=g) / d ** 0.5
    for k, dtype in ((64, torch.bfloat16), (32, torch.float32), (33, torch.float32)):
        qq, kk = q.to(dtype), keys.to(dtype)
        vals, idx = pkg.knn_topk(qq, kk, k, normalize=True)
        check_topk(qq, kk, vals, idx, k, True, EPS[dtype])


def test_imagenet_shape_sampled_rows(pkg):
    """4096 queries against 1 281 167 keys at d = 768 (bf16): fp64 check of a sample of rows, and no buffer of
    size N_q x N_k (4096 x 1.28M fp32 would be 21 GB)."""
    n_q, n_k, d, k = 4096, 1281167, 768, 20
    q, keys = unit(n_q, d, 41, torch.bfloat16), unit(n_k, d, 42, torch.bfloat16)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    vals, idx = pkg.knn_topk(q, keys, k, normalize=True)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    # norms (fp32 copies of the operands while they are summed: 3.9 GB for the keys) and O(N_q k + N_k) scratch
    assert extra < 6 * 2 ** 30, extra
    g = torch.Generator(device="cuda").manual_seed(43)
    rows = torch.randperm(n_q, device="cuda", generator=g)[:192]
    check_topk(q, keys, vals, idx, k, True, EPS[torch.bfloat16], rows=rows, block=64)
    print(f"[knn] 4096 x 1281167 d=768 bf16: extra peak {extra / 2 ** 20:.0f} MiB")


def test_side_stream_and_graph_capture(pkg):
    q, keys = unit(600, 512, 51, torch.float32), unit(7000, 512, 52, torch.float32)
    v0, i0 = pkg.knn_topk(q, keys, 20, normalize=True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        v1, i1 = pkg.knn_topk(q, keys, 20, normalize=True)  # also warms up the capture below
    s.synchronize()
    assert torch.equal(v0, v1) and torch.equal(i0, i1)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gv, gi = pkg.knn_topk(q, keys, 20, normalize=True)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(gv, v0) and torch.equal(gi, i0)


def clustered(n, d, centres, labels_gen, noise):
    y = torch.randint(0, centres.shape[0], (n,), device="cuda", generator=labels_gen)
    x = centres[y] + noise * torch.randn(n, d, device="cuda", generator=labels_gen) / d ** 0.5
    return x, y


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_classify_against_restatement(pkg, dtype):
    """Equal top-1 / top-5 counts, up to the queries whose neighbour set itself is decided by a near-tie at the k-th
    score (the kernel's set differs from the fp64 one): only those may vote differently."""
    c, d = 1000, 256
    centres = unit(c, d, 61, torch.float32)
    g = torch.Generator(device="cuda").manual_seed(62)
    xtr, ytr = clustered(50000, d, centres, g, 3.0)
    xte, yte = clustered(3000, d, centres, g, 3.0)
    xtr, xte = xtr.to(dtype), xte.to(dtype)
    got = pkg.knn_classify(xtr, ytr, xte, yte, k=(10, 20), T=0.07, num_classes=c)
    want = knn_classify_ref(xtr, ytr, xte, yte, k=(10, 20), T=0.07, num_classes=c)
    assert list(got) == ["knn_top1@10", "knn_top5@10", "knn_top1@20", "knn_top5@20"]
    assert all(isinstance(v, float) for v in got.values())
    _, idx = pkg.knn_topk(xte, xtr, 20, normalize=True)
    _, ref_idx = knn_topk_ref(xte, xtr, 20, normalize=True)
    n = xte.shape[0]
    for k in (10, 20):
        differ = int((idx[:, :k].sort(1).values != ref_idx[:, :k].sort(1).values).any(1).sum())
        for key in (f"knn_top1@{k}", f"knn_top5@{k}"):
            assert abs(got[key] - want[key]) * n / 100.0 <= differ + 1e-6, (key, got[key], want[key], differ)
        print(f"[knn] classify {dtype} k={k}: {got[f'knn_top1@{k}']:.2f} / {got[f'knn_top5@{k}']:.2f} % "
              f"(restatement {want[f'knn_top1@{k}']:.2f} / {want[f'knn_top5@{k}']:.2f}), {differ} neighbour sets "
              "differ from fp64")
    assert 5.0 < got["knn_top1@20"] < 99.0  # the data is neither trivial nor noise
    for k in (10, 20):
        one = pkg.knn_classify(xtr, ytr, xte, yte, k=k, num_classes=c)
        assert one == {key: v for key, v in got.items() if key.endswith(f"@{k}")}
    inferred = pkg.knn_classify(xtr, ytr.int(), xte, yte.int(), k=(10, 20))  # C from the labels, int32 labels
    assert inferred == pkg.knn_classify(xtr, ytr, xte, yte, k=(10, 20),
                                        num_classes=int(max(ytr.max(), yte.max())) + 1)


def test_errors_on_device(pkg):
    q, keys = unit(10, 64, 71, torch.float32), unit(40, 64, 72, torch.float32)
    with pytest.raises(ValueError, match="exceeds the number of keys"):
        pkg.knn_topk(q, keys, 41)
    with pytest.raises(ValueError, match=r"k must lie in \[1, 64\]"):
        pkg.knn_topk(q, unit(100, 64, 73, torch.float32), 65)
    y = (torch.arange(40, device="cuda") % 4)
    bad = y.clone()
    bad[7] = 4
    with pytest.raises(ValueError, match="must lie in"):
        pkg.knn_classify(keys, bad, q, y[:10], k=5, num_classes=4)
    with pytest.raises(ValueError, match="must lie in"):
        pkg.knn_classify(keys, y, q, -y[:10] - 1, k=5)
    with pytest.raises(ValueError, match="one entry per feature row"):
        pkg.knn_classify(keys, y[:39], q, y[:10], k=5)
