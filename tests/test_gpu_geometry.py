"""Embedding geometry (geometry.py -> dsoft_geometry -> dsoft_fwd_kernel<MODE_GEOM> + the positives' pre-pass)
against the fp64 restatement in tests/geometry_ref.py, computed on the GPU in row blocks.

Rule, with eps = 2e-5 for split fp32 / fp16 inputs and 4e-6 for bf16 inputs (the cosine accuracy of retrieval and kNN):
  * uniformity: |U - U_fp64| <= 2 t eps + 1e-6 (dU / dcos_ij is 2 t times weights that sum to 1);
  * histograms: the totals are exact, and the number of pairs on the low side of every bin edge (below, then each
    bin, cumulated) differs from the fp64 count by at most the pairs whose fp64 cosine lies within eps of that edge;
  * anisotropy: within 1e-9 of the closed form over the same scaled rows (hi + lo of a split, fp32 1 / ||row||), and
    within 2 eps of the fp64 one;
  * alignment: at alpha = 2 within 2 eps + 1e-6 of fp64; other alpha against the restatement evaluated on the
    positives' cosines the kernel computed.
Unit rows with entries +-1/4 at d = 16 make every cosine an exact multiple of 1/8: there the counts must equal the fp64
assignment exactly, edges and the closed last bin included."""
import math

import pytest
import torch

from geometry_ref import alignment_ref, embedding_geometry_ref, image_text_geometry_ref

pytestmark = pytest.mark.gpu

EPS = {torch.float32: 2e-5, torch.float16: 2e-5, torch.bfloat16: 4e-6}


def rows(n, d, seed, dtype, spread=None, centres=64):
    """Random rows (norms away from 1), or clustered ones (spread: noise around `centres` unit directions)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    if spread is None:
        x = torch.randn(n, d, device="cuda", generator=g) * (0.5 + 2 * torch.rand(n, 1, device="cuda", generator=g))
    else:
        c = torch.nn.functional.normalize(torch.randn(centres, d, device="cuda", generator=g), dim=1)
        x = c[torch.randint(0, centres, (n,), device="cuda", generator=g)] + spread * torch.randn(
            n, d, device="cuda", generator=g) / d ** 0.5
    return x.to(dtype)


def check_hist(hist, below, above, ref_hist, ref_near):
    bins = ref_hist.numel() - 2
    got = torch.cat([torch.tensor([below]), hist, torch.tensor([above])]).to(torch.int64)
    want = torch.cat([ref_hist[bins:bins + 1], ref_hist[:bins], ref_hist[bins + 1:]]).cpu()
    assert int(got.sum()) == int(want.sum())
    diff = (got.cumsum(0)[:-1] - want.cumsum(0)[:-1]).abs()  # low side of edge 0 (lo), 1, .., bins (hi)
    assert bool((diff <= ref_near.cpu()).all()), (diff.max(), got, want)
    return int((got - want).abs().sum())


def scaled_rows(pkg, x):
    """x^_i = r_i x_i in fp64 over the values the kernel multiplies (the statement of the closed-form anisotropy)."""
    from dinosoft_b200.geometry import _prepare

    a, _, _, r, _, dp, lo_at = _prepare(x, x, torch.device("cuda"))
    v = a[:, :dp].double()
    if lo_at is not None:
        v = v + a[:, lo_at:lo_at + dp].double()
    return v * r.double()[:, None]


# (n, d, dtype, t, bins, clustered): every N of {2, 3, 255, 257, 4096, 5003}, d of {8, 512, 768}, each input dtype
CASES = [
    (2, 8, torch.float32, 2.0, 10, False),
    (3, 512, torch.bfloat16, 2.0, 100, False),
    (3, 768, torch.float16, 1.0, 0, False),
    (255, 768, torch.float32, 2.0, 256, True),
    (255, 8, torch.bfloat16, 5.0, 7, False),
    (257, 512, torch.float16, 2.0, 100, True),
    (257, 768, torch.bfloat16, 20.0, 50, True),
    (4096, 512, torch.float32, 2.0, 100, True),
    (4096, 8, torch.float16, 0.5, 64, True),
    (5003, 768, torch.bfloat16, 2.0, 100, True),
    (5003, 512, torch.float32, 3.0, 32, False),
]


@pytest.mark.parametrize("n, d, dtype, t, bins, clustered", CASES)
def test_embedding_geometry_against_fp64(pkg, n, d, dtype, t, bins, clustered):
    x = rows(n, d, n * 13 + d, dtype, spread=1.0 if clustered else None)
    eps = EPS[dtype]
    got = pkg.embedding_geometry(x, t=t, bins=bins)
    ref = embedding_geometry_ref(x, t=t, bins=bins, eps=eps)
    assert isinstance(got["uniformity"], float) and isinstance(got["anisotropy"], float)
    du = abs(got["uniformity"] - ref["uniformity"])
    assert du <= 2 * t * eps + 1e-6, du
    xh = scaled_rows(pkg, x)
    s = xh.sum(0)
    aniso_same = float((s @ s - (xh * xh).sum()) / (n * (n - 1)))
    assert abs(got["anisotropy"] - aniso_same) <= 1e-9
    assert abs(got["anisotropy"] - ref["anisotropy"]) <= 2 * eps
    moved = 0
    if bins:
        assert got["hist"].dtype == torch.int64 and got["hist"].device.type == "cpu" and got["hist"].shape == (bins,)
        assert int(got["hist"].sum()) + got["below"] + got["above"] == n * (n - 1) // 2
        moved = check_hist(got["hist"], got["below"], got["above"], ref["hist"], ref["near"])
    else:
        assert "hist" not in got
    print(f"[geometry] {n}x{d} {dtype} t={t}: |dU| {du:.1e}, U {got['uniformity']:.5f}, aniso "
          f"{got['anisotropy']:.5f}, {moved} counts moved across edges")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("n", [300, 2000])
def test_exact_cosines_on_bin_edges(pkg, dtype, n):
    """Unit rows of +-1/4 at d = 16: cosines are exact multiples of 1/8 and land on the edges of 1/16-wide bins."""
    g = torch.Generator(device="cuda").manual_seed(n)
    base = torch.randint(0, 2, (256, 16), device="cuda", generator=g).float() * 0.5 - 0.25
    x = base[torch.randint(0, 256, (n,), device="cuda", generator=g)].to(dtype)  # repeated rows: cosines of 1
    got = pkg.embedding_geometry(x, t=2.0, bins=32)
    ref = embedding_geometry_ref(x, t=2.0, bins=32)
    assert got["hist"].tolist() == ref["hist"][:32].tolist()
    assert (got["below"], got["above"]) == (0, 0) == (int(ref["hist"][32]), int(ref["hist"][33]))
    assert int(got["hist"][-1]) > 0  # cos == 1 (equal rows) sits on hi: the closed last bin
    # a narrower range: +-1 fall outside it, and edges at multiples of 1/8 again
    got = pkg.embedding_geometry(x, t=2.0, bins=12, range=(-0.75, 0.75))
    ref = embedding_geometry_ref(x, t=2.0, bins=12, range=(-0.75, 0.75))
    assert got["hist"].tolist() == ref["hist"][:12].tolist()
    assert (got["below"], got["above"]) == (int(ref["hist"][12]), int(ref["hist"][13]))
    assert abs(got["uniformity"] - ref["uniformity"]) <= 1e-6


# (n_img, n_txt, d, dtype, captions per image or None (1:1))
PAIR_CASES = [
    (2, 2, 8, torch.float32, None),
    (257, 257, 512, torch.float32, None),
    (4096, 4096, 768, torch.bfloat16, None),
    (1000, 5003, 512, torch.float16, 5),
    (255, 1275, 768, torch.bfloat16, 5),
    (3001, 9003, 8, torch.float32, 3),
]


@pytest.mark.parametrize("n_img, n_txt, d, dtype, per", PAIR_CASES)
def test_image_text_geometry_against_fp64(pkg, n_img, n_txt, d, dtype, per):
    img = rows(n_img, d, n_img + d, dtype, spread=1.0)
    tmap = None
    if per is None:
        txt = (img.float() + 0.5 * rows(n_txt, d, n_txt + 1, torch.float32, spread=1.0)).to(dtype)
    else:
        g = torch.Generator(device="cuda").manual_seed(n_txt)
        tmap = torch.arange(n_txt, device="cuda")[torch.randperm(n_txt, device="cuda", generator=g)] % n_img
        txt = (img.float()[tmap] + 0.5 * rows(n_txt, d, n_txt + 1, torch.float32, spread=1.0)).to(dtype)
    eps = EPS[dtype]
    got = pkg.image_text_geometry(img, txt, tmap, bins=100)
    ref = image_text_geometry_ref(img, txt, tmap, bins=100, eps=eps)
    assert isinstance(got["alignment"], float)
    assert abs(got["alignment"] - ref["alignment"]) <= 2 * eps + 1e-6
    assert int(got["pos_hist"].sum()) + got["pos_below"] + got["pos_above"] == n_txt
    assert int(got["neg_hist"].sum()) + got["neg_below"] + got["neg_above"] == n_img * n_txt - n_txt
    moved = check_hist(got["pos_hist"], got["pos_below"], got["pos_above"], ref["pos_hist"], ref["pos_near"])
    moved += check_hist(got["neg_hist"], got["neg_below"], got["neg_above"], ref["neg_hist"], ref["neg_near"])
    print(f"[geometry] {n_img}x{n_txt} d={d} {dtype}: alignment {got['alignment']:.6f} (fp64 {ref['alignment']:.6f}),"
          f" {moved} counts moved across edges")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_alignment_other_alpha_on_kernel_cosines(pkg, dtype):
    from dinosoft_b200.geometry import _prepare, _run

    img = rows(700, 512, 81, dtype, spread=1.0)
    g = torch.Generator(device="cuda").manual_seed(82)
    tmap = torch.arange(2100, device="cuda") % 700
    txt = (img.float()[tmap] + 0.3 * torch.randn(2100, 512, device="cuda", generator=g) / 512 ** 0.5).to(dtype)
    dev = torch.device("cuda")
    a, b, width, ra, rb, _, _ = _prepare(img, txt, dev)
    t32 = tmap.to(torch.int32)
    ref_cos = image_text_geometry_ref(img, txt, tmap, bins=0)["pos_cos"]
    for alpha in (0.5, 1.0, 3.0):
        sums, _, pos_cos = _run(a, b, width, 700, 2100, ra, rb, t32, 0.0, alpha, -1.0, 1.0, 0, dev, want_pos_cos=True)
        assert float((pos_cos.double() - ref_cos).abs().max()) <= EPS[dtype]
        want = float(alignment_ref(pos_cos, alpha))
        assert float(sums[1]) / 2100 == pytest.approx(want, rel=1e-12)
        assert pkg.image_text_geometry(img, txt, tmap, bins=0, alpha=alpha)["alignment"] == float(sums[1]) / 2100


def test_large_pool_no_quadratic_memory(pkg):
    """158 915 x 512 fp32 (Flickr30k's caption count), clustered: against the chunked fp64 restatement, and nothing of
    size N^2 allocated (the fp32 distances of the pdist recipe alone are 50 GB)."""
    n, d = 158915, 512
    x = rows(n, d, 91, torch.float32, spread=0.8, centres=1000)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    got = pkg.embedding_geometry(x, t=2.0, bins=100)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    # split operands (2 x 3 x 2 bytes per feature), fp32 / fp64 norm and anisotropy chunks, O(N) scratch
    assert extra < 4 * 2 ** 30, extra
    ref = embedding_geometry_ref(x, t=2.0, bins=100, eps=EPS[torch.float32], block=4096)
    du = abs(got["uniformity"] - ref["uniformity"])
    assert du <= 4 * EPS[torch.float32] + 1e-6
    assert abs(got["anisotropy"] - ref["anisotropy"]) <= 2 * EPS[torch.float32]
    moved = check_hist(got["hist"], got["below"], got["above"], ref["hist"], ref["near"])
    print(f"[geometry] {n}x{d} fp32: extra peak {extra / 2 ** 20:.0f} MiB, |dU| {du:.1e}, {moved} counts moved")


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32, torch.bfloat16])
def test_noncontiguous_and_host_inputs(pkg, dtype):
    big = rows(600, 2 * 264, 101, dtype, spread=1.0)
    x = big[:, ::2]                        # strided columns
    assert not x.is_contiguous()
    want = pkg.embedding_geometry(x.contiguous(), bins=40)
    got = pkg.embedding_geometry(x.cpu(), bins=40)  # a host tensor is copied to the device
    assert got["uniformity"] == want["uniformity"] and got["anisotropy"] == want["anisotropy"]
    assert torch.equal(got["hist"], want["hist"])
    txt = rows(900, 264, 102, dtype, spread=1.0).t().contiguous().t()  # column-major
    tmap = torch.arange(900) % 600
    a = pkg.image_text_geometry(x.cpu(), txt.cpu(), tmap)
    b = pkg.image_text_geometry(x.contiguous(), txt.contiguous(), tmap.cuda())
    assert a["alignment"] == b["alignment"] and torch.equal(a["neg_hist"], b["neg_hist"])


def test_repeatable_side_stream_and_graph_capture(pkg):
    from dinosoft_b200.geometry import _prepare, _run

    x = rows(6000, 512, 111, torch.float32, spread=1.0)
    r0, r1 = pkg.embedding_geometry(x, bins=100), pkg.embedding_geometry(x, bins=100)
    assert r0["uniformity"] == r1["uniformity"] and torch.equal(r0["hist"], r1["hist"])  # bit-identical
    dev = torch.device("cuda")
    img, txt = rows(3000, 256, 112, torch.bfloat16, spread=1.0), rows(7000, 256, 113, torch.bfloat16, spread=1.0)
    tmap = (torch.arange(7000, device="cuda") % 3000).to(torch.int32)
    a, b, width, ra, _, _, _ = _prepare(x, x, dev)
    ia, ib, iw, ira, irb, _, _ = _prepare(img, txt, dev)

    def both():
        one = _run(a, b, width, 6000, 0, ra, None, None, 2.0, 1.0, -1.0, 1.0, 100, dev)
        two = _run(ia, ib, iw, 3000, 7000, ira, irb, tmap, 0.0, 2.0, -1.0, 1.0, 64, dev)
        return one[0], one[1], two[0], two[1]

    eager = [t.clone() for t in both()]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        side = both()  # also warms up the capture below
    s.synchronize()
    assert all(torch.equal(u, v) for u, v in zip(eager, side))
    assert float(eager[0][0]) > 0 and int(eager[3].sum()) == 3000 * 7000
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = both()
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(u, v) for u, v in zip(eager, captured))


def test_einval_through_the_abi(pkg):
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    assert lib.dsoft_geometry_scratch_bytes(1000, 0, 100) > 0 and lib.dsoft_geometry_scratch_bytes(10, 30, 256) > 0
    assert lib.dsoft_geometry_scratch_bytes(1000, 0, 257) == 0
    x = torch.zeros(64, 8, dtype=torch.bfloat16, device="cuda")
    sums = torch.zeros(2, dtype=torch.float64, device="cuda")
    hist = torch.zeros(2, 12, dtype=torch.int64, device="cuda")
    scratch = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    p = lambda t: t.data_ptr()
    args = [p(x), None, 8, 64, 0, None, None, None, 2.0, 2.0, -1.0, 1.0, 10, p(sums), p(hist), None, p(scratch), None]
    assert lib.dsoft_geometry(*args) == 0
    torch.cuda.synchronize()
    assert int(hist[0].sum()) == 64 * 63 // 2 and int(hist[0, 5]) == 64 * 63 // 2  # zero rows: cosine 0
    assert float(sums[0]) == pytest.approx(64 * 63 / 2 * math.exp(-4.0), rel=1e-6)
    for i, bad in [(8, 21.0), (12, 300), (2, 12), (3, 1), (10, 1.0)]:
        a = list(args)
        a[i] = bad
        if i == 10:  # lo == hi
            a[11] = 1.0
        assert lib.dsoft_geometry(*a) == -1, (i, bad)
        assert lib.dsoft_last_error()
    with pytest.raises(ValueError, match="at least 2 rows"):
        pkg.embedding_geometry(x[:1])
