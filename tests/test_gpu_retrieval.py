"""Retrieval ranks and R@K (retrieval.py -> dsoft_retrieval_ranks -> dsoft_fwd_kernel<MODE_RANKS>) against an fp64
statement of the counts, computed on the GPU in row blocks.

Rule: a query's rank may differ from the fp64 count only by the number of its non-positive scores that lie within
eps of its threshold (eps = 2e-5 for split fp32 / fp16 inputs, 4e-6 for bf16 inputs, unit-norm features).  Integer
features make every score exact, and the ranks then have to match exactly, ties included."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

EPS = {torch.float32: 2e-5, torch.float16: 2e-5, torch.bfloat16: 4e-6}


def fp64_counts(img, txt, tmap=None, eps=0.0, block=4096):
    """Exact ranks in fp64 plus, per query, how many non-positive scores lie within eps of its threshold.  Row blocks
    of `block` images: O(block * N_txt) memory."""
    dev = torch.device("cuda")
    a, b = img.to(dev, torch.float64), txt.to(dev, torch.float64)
    n_img, n_txt = a.shape[0], b.shape[0]
    t = torch.arange(n_txt, device=dev) if tmap is None else tmap.to(dev, torch.int64)
    thr_txt = (a[t] * b).sum(1)  # s_t(j),j
    p = torch.full((n_img,), -float("inf"), dtype=torch.float64, device=dev).scatter_reduce(0, t, thr_txt, "amax")
    rank_img = torch.zeros(n_img, dtype=torch.int64, device=dev)
    near_img = torch.zeros_like(rank_img)
    rank_txt = torch.zeros(n_txt, dtype=torch.int64, device=dev)
    near_txt = torch.zeros_like(rank_txt)
    for r0 in range(0, n_img, block):
        s = a[r0:r0 + block] @ b.t()
        rows = torch.arange(r0, r0 + s.shape[0], device=dev)
        other = t[None, :] != rows[:, None]
        pr = p[r0:r0 + s.shape[0], None]
        rank_img[r0:r0 + s.shape[0]] = (other & (s > pr)).sum(1)
        near_img[r0:r0 + s.shape[0]] = (other & ((s - pr).abs() <= eps)).sum(1)
        rank_txt += (other & (s > thr_txt[None, :])).sum(0)
        near_txt += (other & ((s - thr_txt[None, :]).abs() <= eps)).sum(0)
        del s, other
    return rank_img, rank_txt, near_img, near_txt


def check_ranks(got, want, near, label):
    """|got - want| <= near per query; returns the number of queries that differ."""
    diff = (got.to(want.device) - want).abs()
    bad = diff > near
    assert not bool(bad.any()), (label, int(bad.sum()), diff[bad][:8].tolist(), near[bad][:8].tolist())
    return int((diff > 0).sum())


def flip_distance(img, txt, got, want, idx_img=True):
    """Largest distance between a flipped query's threshold and the score that explains its flip (the |diff|-th
    closest non-positive score): what the eps of the rule has to cover on this data.  1:1 pools only."""
    a, b = img.cuda().double(), txt.cuda().double()
    diff = (got.cuda() - want.cuda()).abs()
    worst = 0.0
    for q in torch.nonzero(diff).flatten().tolist():
        s = (a[q] @ b.t()) if idx_img else (a @ b[q])
        d = (s - s[q]).abs()
        d[q] = float("inf")
        worst = max(worst, float(d.sort().values[int(diff[q]) - 1]))
    return worst


def get_clip_metrics(image_features, text_features, logit_scale):
    """open_clip 2.31.0 open_clip_train/train.py get_clip_metrics, as written there."""
    metrics = {}
    logits_per_image = (logit_scale * image_features @ text_features.t()).detach().cpu()
    logits_per_text = logits_per_image.t().detach().cpu()
    logits = {"image_to_text": logits_per_image, "text_to_image": logits_per_text}
    ground_truth = torch.arange(len(text_features)).view(-1, 1)
    for name, logit in logits.items():
        ranking = torch.argsort(logit, descending=True)
        preds = torch.where(ranking == ground_truth)[1]
        preds = preds.detach().cpu().numpy()
        metrics[f"{name}_mean_rank"] = preds.mean() + 1
        metrics[f"{name}_median_rank"] = np.floor(np.median(preds)) + 1
        for k in [1, 5, 10]:
            metrics[f"{name}_R@{k}"] = np.mean(preds < k)
    return metrics


def pool(n_img, n_txt, d, seed, tmap=None, noise=15.0):
    """Unit-norm features; caption j is image t(j) plus noise of norm ~noise: the positive's score (~1/noise) sits
    about 1.5 standard deviations of the negatives' (~d^-1/2) above them, so the ranks spread over hundreds and many
    scores lie close to a threshold."""
    g = torch.Generator().manual_seed(seed)
    img = torch.nn.functional.normalize(torch.randn(n_img, d, generator=g, dtype=torch.float64), dim=-1)
    t = torch.arange(n_txt) if tmap is None else tmap
    txt = torch.nn.functional.normalize(img[t] + noise * torch.randn(n_txt, d, generator=g, dtype=torch.float64)
                                        / d ** 0.5, dim=-1)
    return img.float(), txt.float()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n", [1, 2, 255, 256, 257, 4133])
def test_square_pool(pkg, n, dtype):
    img, txt = pool(n, n, 512, seed=n)
    img, txt = img.to(dtype), txt.to(dtype)
    ri, rt = pkg.retrieval_ranks(img.cuda(), txt.cuda())
    assert ri.dtype == rt.dtype == torch.int64 and ri.shape == (n,) and rt.shape == (n,) and ri.is_cuda
    wi, wt, ni, nt = fp64_counts(img, txt, eps=EPS[dtype])
    flips = check_ranks(ri, wi, ni, "img") + check_ranks(rt, wt, nt, "txt")
    dist = max(flip_distance(img, txt, ri, wi, True), flip_distance(img, txt, rt, wt, False)) if flips else 0.0
    print(f"[retrieval] n={n} {dtype}: R@1 i2t {float((ri == 0).float().mean()):.4f}, median rank "
          f"{float(ri.float().median()):.0f}, {flips} flipped ranks, largest flip distance {dist:.2e}")
    got = pkg.clip_metrics(img.cuda(), txt.cuda(), logit_scale=torch.tensor(100.0))
    if flips == 0:
        want = get_clip_metrics(img.double().cuda(), txt.double().cuda(), 100.0)
        assert list(got) == list(want)
        for key in want:
            assert got[key] == float(want[key]), (key, got[key], want[key])


def caption_map(n_img, counts, seed):
    g = torch.Generator().manual_seed(seed)
    t = torch.repeat_interleave(torch.arange(n_img), counts)
    return t[torch.randperm(t.numel(), generator=g)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_five_captions_per_image(pkg, dtype):
    tm = caption_map(1000, torch.full((1000,), 5), seed=1)
    img, txt = pool(1000, 5000, 768, seed=2, tmap=tm)
    img, txt = img.to(dtype), txt.to(dtype)
    ri, rt = pkg.retrieval_ranks(img.cuda(), txt.cuda(), tm.cuda())
    wi, wt, ni, nt = fp64_counts(img, txt, tm, eps=EPS[dtype])
    flips = check_ranks(ri, wi, ni, "img") + check_ranks(rt, wt, nt, "txt")
    print(f"[retrieval] 1000 x 5000 {dtype}: R@1 i2t {float((ri == 0).float().mean()):.4f}, {flips} flipped ranks")
    from dinosoft_b200.retrieval import metrics_from_ranks

    m = pkg.clip_metrics(img, txt, text_image=tm)  # host tensors: copied to the device
    assert m == metrics_from_ranks(ri, rt)  # integer counts: the same ranks on every call


def test_one_to_seven_captions(pkg):
    g = torch.Generator().manual_seed(3)
    counts = torch.randint(1, 8, (700,), generator=g)
    counts[:2] = torch.tensor([1, 7])
    tm = caption_map(700, counts, seed=4)
    img, txt = pool(700, int(counts.sum()), 256, seed=5, tmap=tm)
    ri, rt = pkg.retrieval_ranks(img, txt, tm.to(torch.int32))
    wi, wt, ni, nt = fp64_counts(img, txt, tm, eps=EPS[torch.float32])
    check_ranks(ri, wi, ni, "img")
    check_ranks(rt, wt, nt, "txt")


@pytest.mark.parametrize("d", [500, 512, 768, 1024])
def test_fp16_noncontiguous_widths(pkg, d):
    img, txt = pool(777, 777, d, seed=d)
    img16 = img.half().cuda()
    txt_nc = torch.cat([txt, txt], dim=1).cuda()[:, :d]  # non-contiguous view (row stride 2 d), same values
    assert not txt_nc.is_contiguous()
    ri, rt = pkg.retrieval_ranks(img16, txt_nc)
    wi, wt, ni, nt = fp64_counts(img16.float(), txt, eps=EPS[torch.float16])
    check_ranks(ri, wi, ni, "img")
    check_ranks(rt, wt, nt, "txt")
    # column-major fp32 images against bf16 texts: both sides take the split form (bf16 with a zero lo part)
    img_cm = img.cuda().t().contiguous().t()
    assert not img_cm.is_contiguous()
    ri2, rt2 = pkg.retrieval_ranks(img_cm, txt.cuda().bfloat16())
    wi, wt, ni, nt = fp64_counts(img, txt.bfloat16().float(), eps=EPS[torch.float32])
    check_ranks(ri2, wi, ni, "img mixed")
    check_ranks(rt2, wt, nt, "txt mixed")


@pytest.mark.parametrize("n_img, n_txt, mapped", [(300, 300, False), (257, 257, False), (1, 1, False),
                                                    (131, 523, True), (256, 1031, True)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_exact_ties_integer_features(pkg, n_img, n_txt, mapped, dtype):
    """Small integer features: every score is an exact integer in any summation order, so ties are exact and the
    kernel must reproduce the strict-> count exactly (not argsort's arbitrary order).  Duplicated caption rows
    tie with the positive; duplicated image rows tie across queries."""
    g = torch.Generator().manual_seed(n_img * 7 + n_txt)
    img = torch.randint(-3, 4, (n_img, 64), generator=g).float()
    txt = torch.randint(-3, 4, (n_txt, 64), generator=g).float()
    tm = None
    if mapped:
        tm = torch.cat([torch.arange(n_img), torch.randint(0, n_img, (n_txt - n_img,), generator=g)])
    if n_txt > 10:
        txt[9] = txt[5]
        img[min(7, n_img - 1)] = img[min(3, n_img - 1)]
    ri, rt = pkg.retrieval_ranks(img.to(dtype).cuda(), txt.to(dtype).cuda(), None if tm is None else tm.cuda())
    wi, wt, _, _ = fp64_counts(img, txt, tm)
    assert torch.equal(ri, wi) and torch.equal(rt, wt)
    if n_txt > 10 and not mapped:  # the duplicated caption ties with image 5's positive: not counted
        s = img[5].double() @ txt.double().t()
        assert s[9] == s[5] and int(ri[5]) == int((s > s[5]).sum())


def test_65536_pool_no_square_buffer(pkg):
    n, d = 65536, 256
    img, txt = pool(n, n, d, seed=65536)
    img, txt = img.cuda(), txt.cuda()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    ri, rt = pkg.retrieval_ranks(img, txt)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    # split operands 2 x 3 x n x d bf16 (200 MB), their hi / lo parts while they are built (134 MB) and O(n)
    # vectors; one byte per pair would be 4.3 GB
    assert extra < 512 * 2 ** 20, extra
    wi, wt, ni, nt = fp64_counts(img, txt, eps=EPS[torch.float32], block=2048)
    flips = check_ranks(ri, wi, ni, "img") + check_ranks(rt, wt, nt, "txt")
    print(f"[retrieval] 65536^2 fp32: extra peak {extra / 2 ** 20:.1f} MiB, median rank {float(ri.float().median()):.0f}, "
          f"{flips} flipped ranks")


def test_side_stream_and_graph_capture(pkg):
    tm = caption_map(600, torch.full((600,), 3), seed=6)
    img, txt = pool(600, 1800, 512, seed=7, tmap=tm)
    img, txt, tm = img.cuda(), txt.cuda(), tm.cuda()
    ri, rt = pkg.retrieval_ranks(img, txt, tm)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ri2, rt2 = pkg.retrieval_ranks(img, txt, tm, check=False)  # also warms up the capture below
    s.synchronize()
    assert torch.equal(ri, ri2) and torch.equal(rt, rt2)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gi, gt = pkg.retrieval_ranks(img, txt, tm, check=False)
    for _ in range(2):  # replays rewrite (not accumulate) the ranks
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(gi, ri) and torch.equal(gt, rt)


def test_errors_on_device(pkg):
    img, txt = pool(50, 100, 64, seed=8, tmap=torch.arange(100) % 50)
    img, txt = img.cuda(), txt.cuda()
    with pytest.raises(ValueError, match="pass text_image"):
        pkg.retrieval_ranks(img, txt)
    bad = (torch.arange(100) % 50).cuda()
    bad[17] = 50
    with pytest.raises(ValueError, match="must lie in"):
        pkg.clip_metrics(img, txt, text_image=bad)
    nocap = (torch.arange(100) % 49).cuda()
    with pytest.raises(ValueError, match="have no text"):
        pkg.retrieval_ranks(img, txt, nocap)
