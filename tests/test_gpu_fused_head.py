"""Fused projection head (SURVEY 8f-3, dsoft_head_forward): under bf16 autocast the Linear / Linear-ReLU-Linear head
runs on the tcgen05 tile kernel and writes the student columns of the packed buffer.  Checked against the PyTorch
head under the same autocast (the arithmetic the reference gets at train.py:285): bf16 outputs may differ by one
rounding step on isolated elements, nothing more.  The kernel alone is checked against the fp64 autocast reference
(tests/autocast_head_ref.py) at every rank position, on both tile schedules; the module under autocast against fp64
is tests/test_gpu_autocast_head.py."""
import ctypes as C

import pytest
import torch

from gpu_util import make_args, rel_err, synth

pytestmark = pytest.mark.gpu


def _run(pkg, img, txt, dino, args, fused, seed=3, **ctor):
    from dinosoft_b200 import loss as loss_mod

    old = loss_mod.FUSED_HEAD
    loss_mod.FUSED_HEAD = fused
    try:
        dev = "cuda"
        loss = pkg.ClipLossWithDINOEnhancements(**ctor)
        torch.manual_seed(seed)
        loss.init_proj(img.shape[1], dino.shape[1], dev, args.projection_type)
        im = img.to(dev).requires_grad_(True)
        tx = txt.to(dev).requires_grad_(True)
        sc = torch.tensor(25.0, device=dev, requires_grad=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = loss(im, tx, sc, dino.to(dev), args, output_dict=True)
        out["total_loss"].backward()
        torch.cuda.synchronize()
        grads = {n: p.grad.detach().clone() for n, p in loss.image_to_dino_proj.named_parameters()}
        return out, im.grad, tx.grad, sc.grad, grads
    finally:
        loss_mod.FUSED_HEAD = old


@pytest.mark.parametrize("ptype", ["mlp", "linear"])
@pytest.mark.parametrize("B,D,Dd", [(512, 128, 192), (1000, 512, 768), (300, 72, 136)])
def test_fused_head_matches_autocast_head(pkg, ptype, B, D, Dd):
    img, txt, dino = synth(17, B, D, Dd)
    args = make_args(use_projection=True, projection_type=ptype)
    o1, gi1, gt1, gs1, gh1 = _run(pkg, img, txt, dino, args, True)
    o0, gi0, gt0, gs0, gh0 = _run(pkg, img, txt, dino, args, False)
    for k in ("total_loss", "classic_loss", "soft_loss"):
        a, b = float(o1[k]), float(o0[k])
        print(f"[fused head {ptype}] {k}: fused {a:.6f} torch {b:.6f}")
        # isolated one-step bf16 differences of the student move the soft term at the 1e-4 level
        assert a == pytest.approx(b, rel=1e-3), k
    assert float(o1["classic_loss"]) == pytest.approx(float(o0["classic_loss"]), rel=1e-6)
    for name, a, b in (("d_image", gi1, gi0), ("d_text", gt1, gt0)):
        linf, l2 = rel_err(a, b)
        print(f"[fused head {ptype}] {name}: linf={linf:.2e} l2={l2:.2e}")
        assert l2 < 1e-2, (name, linf, l2)
    for n in gh0:
        # the PyTorch path rounds every weight gradient to bf16 (the matmul output dtype under autocast); the
        # fused path keeps the fp32 accumulator, so the comparison is at bf16 resolution
        linf, l2 = rel_err(gh1[n], gh0[n])
        print(f"[fused head {ptype}] d {n}: linf={linf:.2e} l2={l2:.2e}")
        assert l2 < 3e-2, (n, linf, l2)


def _walks_all_tiles(rows, num_sms):
    """launch_linear's schedule rule (dsoft_api.cu, `P.tiles_per_split = (2 * pairs >= p->num_sms) ? ...`): once the
    128-row blocks make 2 * pairs >= num_sms, one CTA pair walks every 256-column tile of its rows."""
    pairs = -(-(-(-rows // 128)) // 2)
    return 2 * pairs >= num_sms


def _schedule_rows(which, num_sms):
    largest_one_tile = 2 * ((num_sms - 1) // 2) * 128  # 18 688 rows on 148 SMs
    return {"one_tile_max": largest_one_tile, "walk_min": largest_one_tile + 1, "b32768": 32768}[which]


_DIMS = {"c1": (512, 640, 768), "small": (128, 160, 192), "ragged": (72, 104, 136), "c4": (768, 896, 1024)}
_HEAD_CASES = [
    # (world, rank, rows b (a multiple of 8 at world > 1) or a schedule size, dims (D, H, Dp) as init_proj makes
    #  them: H = (D + Dd) / 2, Dp = Dd; head type, biases).  Rank 0 of one at b = 700, dims c1, is
    #  test_head_forward_values.
    (2, 1, 696, "c1", "mlp", True),
    (8, 7, 136, "small", "mlp", True),
    (8, 3, 136, "small", "mlp", True),
    (4, 3, 296, "ragged", "mlp", True),
    (2, 0, 296, "ragged", "mlp", False),
    (1, 0, 256, "c4", "mlp", True),
    (4, 2, 256, "c4", "mlp", True),
    (1, 0, 300, "ragged", "linear", True),
    (8, 7, 296, "ragged", "linear", True),
    (2, 1, 296, "ragged", "linear", False),
    (4, 3, 696, "c1", "linear", True),
    (1, 0, "one_tile_max", "c1", "mlp", True),
    (1, 0, "walk_min", "c1", "mlp", True),
    (2, 1, "walk_min", "c1", "mlp", True),
    (1, 0, "b32768", "c1", "mlp", True),
]


def test_head_forward_values(pkg):
    """dsoft_head_forward alone at rank 0 of one, b = 700, D = 512: MLP and Linear head (see _check_head_forward)."""
    _check_head_forward(1, 0, 700, "c1", "mlp", True)
    _check_head_forward(1, 0, 700, "c1", "linear", True)


@pytest.mark.parametrize("W,r,b,dims,ptype,bias", [pytest.param(*c, id=f"w{c[0]}r{c[1]}-{c[2]}-{c[3]}-{c[4]}"
                                                                   + ("" if c[5] else "-nobias"))
                                                   for c in _HEAD_CASES])
def test_head_forward_ranks_and_schedules(pkg, W, r, b, dims, ptype, bias):
    _check_head_forward(W, r, b, dims, ptype, bias)


def _check_head_forward(W, r, b, dims, ptype, bias):
    """dsoft_head_forward alone at rank r of W: the hidden activations and the student columns of this rank's rows
    against the fp64 autocast reference, and nothing else of `gathered` touched (a random bf16 pattern everywhere
    else - other ranks' rows, image / text / DINO columns - must stay bit-identical)."""
    from autocast_head_ref import assert_one_rounding, head_forward, linear_exact
    from dinosoft_b200 import _cabi
    from dinosoft_b200 import loss as loss_mod

    dev = torch.device("cuda", 0)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    if isinstance(b, str):
        which, b = b, _schedule_rows(b, sms)
        if W > 1:  # the plan needs a multiple of 8 here; 18 696 rows still walk all tiles
            b = -(-b // 8) * 8
        assert _walks_all_tiles(b, sms) == (which != "one_tile_max"), (which, b, sms)
    D, H, Dp = _DIMS[dims]
    be = loss_mod._default_backend(dev)
    shape = _cabi.Shape(b=b, world=W, rank=r, D=D, Dp=Dp, Dd=Dp, flags=_cabi.DSOFT_F_SOFT, teacher_temp=0.15,
                        text_temp=0.0, rho=0.1, c_clip=1.0)
    plan = be.plan(shape, dev)
    assert plan.row_elems == 2 * D + 2 * Dp  # image | text | student | DINO, no padding
    g = torch.Generator(device=dev).manual_seed(b + 7 * r + W)
    gathered = (0.5 * torch.randn(W * b, plan.row_elems, generator=g, device=dev)).to(torch.bfloat16)
    before = gathered.clone()
    K1, N1 = (D, H) if ptype == "mlp" else (D, Dp)
    w1 = (torch.randn(N1, K1, generator=g, device=dev) / K1 ** 0.5).to(torch.bfloat16)
    b1 = (0.1 * torch.randn(N1, generator=g, device=dev)) if bias else None
    w2 = b2 = hidden = None
    if ptype == "mlp":
        w2 = (torch.randn(Dp, H, generator=g, device=dev) / H ** 0.5).to(torch.bfloat16)
        b2 = (0.1 * torch.randn(Dp, generator=g, device=dev)) if bias else None
        hbuf = torch.randn(b + 1, H, generator=g, device=dev).to(torch.bfloat16)  # one guard row after `hidden`
        guard = hbuf[b].clone()
        hidden = hbuf[:b]
    be.head_forward(plan, gathered, w1, b1, w2, b2, hidden)
    torch.cuda.synchronize()

    rows = slice(r * b, (r + 1) * b)
    zcols = slice(2 * D, 2 * D + Dp)
    expect = before.clone()
    expect[rows, zcols] = gathered[rows, zcols]
    assert torch.equal(gathered.view(torch.int16), expect.view(torch.int16)), "head forward wrote outside its block"
    x = before[rows, :D]
    if ptype == "mlp":
        assert torch.equal(hbuf[b], guard), "head forward wrote past the hidden rows"
        assert_one_rounding("hidden", hidden, torch.relu(linear_exact(x, w1, b1)))
        # the second layer from the operand the kernel used (its own hidden); both together are
        # autocast_head_ref.head_forward, which the module-level tests use
        assert_one_rounding("student", gathered[rows, zcols], linear_exact(hidden, w2, b2))
        h_ref, _ = head_forward(x, w1, b1, w2, b2)
        assert (hidden.double() != h_ref).double().mean().item() < 0.02  # isolated one-step differences only
    else:
        assert_one_rounding("student", gathered[rows, zcols], linear_exact(x, w1, b1))
