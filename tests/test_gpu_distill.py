"""DistillClipLoss on the B200 (distill.py -> dsoft_distill_forward / _backward -> dsoft_fwd_kernel<MODE_DIST_FWD /
MODE_DIST_G> + the gradient GEMMs) against the fp64 statement of upstream's recipe (tests/distill_ref.py).

Bars: losses 1e-4 relative; d_image / d_text 1e-3 (max error over max magnitude; a bf16 gradient may in addition be
off by its own rounding, 2^-8 of the element - the module returns gradients in the input dtype); d_scale 1e-3
relative.  The backward runs through 0.3 contrastive + 1.7 distill, so that a G which folds g_c = g_d fails.  Inputs
are bf16-representable, so kernel and statement see the same operands."""
import ctypes as C
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT
from gpu_util import rel_err, synth, synth_aligned
import distill_ref

pytestmark = pytest.mark.gpu

LOSS_RTOL, GRAD_RTOL = 1e-4, 1e-3
DEV = "cuda"
EINVAL = -1
GC, GD = 0.3, 1.7


def _inputs(kind, B, D, Dt, seed):
    if kind == "aligned":
        img, txt, _ = synth_aligned(seed, B, D, 8)
        dimg, dtxt, _ = synth_aligned(seed + 1, B, Dt, 8)
    else:
        img, txt, _ = synth(seed, B, D, 8, clustered=(kind == "clustered"))
        dimg, dtxt, _ = synth(seed + 1, B, Dt, 8, clustered=(kind == "clustered"))
    return img.to(DEV), txt.to(DEV), dimg.to(DEV), dtxt.to(DEV)


def _grad_err(got, want, dtype):
    out_round = 2.0 ** -8 if dtype == torch.bfloat16 else 0.0
    excess = (got.double() - want).abs() - out_round * want.abs()
    # B = 1: p = q = 1, so every feature gradient is exactly zero; the floor turns the bar into an absolute one there
    return excess.max().item() / max(want.abs().max().item(), 1e-6)


def _check(pkg, img, txt, dimg, dtxt, s, st, dtype=torch.float32, noncontig=False, gc=GC, gd=GD):
    ref = distill_ref.rank_grads(img.double(), txt.double(), dimg.double(), dtxt.double(), s, st, 1, gc=gc, gd=gd)[0]
    im, tx, di, dx = (t.to(dtype) for t in (img, txt, dimg, dtxt))
    if noncontig:  # every other column of a wider buffer
        def nc(t):
            wide = torch.zeros((t.shape[0], 2 * t.shape[1]), dtype=dtype, device=DEV)
            wide[:, ::2] = t
            return wide[:, ::2]
        im, tx, di, dx = nc(im), nc(tx), nc(di), nc(dx)
        assert not im.is_contiguous() and not di.is_contiguous()
    im, tx = im.detach().requires_grad_(True), tx.detach().requires_grad_(True)
    sc = torch.tensor(float(s), device=DEV, requires_grad=True)
    c, d = pkg.DistillClipLoss()(im, tx, sc, di, dx, torch.tensor(float(st), device=DEV))
    (gc * c + gd * d).backward()
    torch.cuda.synchronize()
    assert c.shape == () and d.shape == () and c.dtype == torch.float32
    assert im.grad.dtype == dtype and tx.grad.dtype == dtype
    for name, got in (("contrastive", c), ("distill", d)):
        assert abs(float(got) - ref[name]) <= LOSS_RTOL * abs(ref[name]), (name, float(got), ref[name])
    for name, got, want in (("d_image", im.grad, ref["d_image"]), ("d_text", tx.grad, ref["d_text"])):
        err = _grad_err(got, want, dtype)
        assert err < GRAD_RTOL, (name, err)
    assert abs(float(sc.grad) - ref["d_scale"]) <= GRAD_RTOL * abs(ref["d_scale"]) + 1e-6, (float(sc.grad),
                                                                                            ref["d_scale"])


# "aligned" (p_ii -> 1) runs at s = 14.29: at s = 50 or 100 synth_aligned's rows are so separated that 1 - p_ii is
# 1e-10 or below fp64 resolution, and the feature gradient itself is below what any fp32 log-sum-exp resolves
CASES = [  # B, (D, Dt), (s, s_t), input kind, dtype, non-contiguous
    (1, (512, 768), (14.29, 100.0), "clustered", torch.float32, False),
    (7, (100, 64), (14.29, 100.0), "aligned", torch.float32, False),   # both widths padded
    (130, (100, 64), (100.0, 100.0), "random", torch.float16, False),
    (300, (512, 768), (50.0, 30.0), "clustered", torch.bfloat16, False),
    (1000, (768, 1024), (14.29, 100.0), "aligned", torch.float16, False),
    (1000, (1024, 512), (50.0, 30.0), "clustered", torch.float32, True),
    (2049, (512, 768), (14.29, 100.0), "aligned", torch.bfloat16, False),
    (4133, (768, 1024), (100.0, 100.0), "random", torch.float16, True),
    (8192, (512, 768), (14.29, 100.0), "clustered", torch.float32, False),
    (8192, (1024, 512), (14.29, 100.0), "aligned", torch.bfloat16, False),
    (8192, (768, 1024), (100.0, 100.0), "clustered", torch.float32, False),
]


@pytest.mark.parametrize("B,dims,ss,kind,dtype,noncontig", CASES)
def test_module_against_fp64(pkg, B, dims, ss, kind, dtype, noncontig):
    img, txt, dimg, dtxt = _inputs(kind, B, dims[0], dims[1], seed=B + dims[0])
    _check(pkg, img, txt, dimg, dtxt, ss[0], ss[1], dtype, noncontig)


@pytest.mark.parametrize("B", [300, 4133])
def test_distill_only_student_near_teacher(pkg, B):
    """Student ~ teacher: d distill / d x = (p - q) terms are small; held to the bar relative to their own magnitude
    (a G formed as fp16(p) - fp16(q) fails this)."""
    D, s = 512, 50.0
    dimg, dtxt, _ = synth(B, B, D, 8)
    dimg, dtxt = dimg.to(DEV), dtxt.to(DEV)
    g = torch.Generator().manual_seed(B + 1)
    r = lambda x: torch.nn.functional.normalize(x, dim=-1).to(torch.bfloat16).float().to(DEV)  # noqa: E731
    img = r(dimg.cpu() + 0.01 * torch.randn(B, D, generator=g))
    txt = r(dtxt.cpu() + 0.01 * torch.randn(B, D, generator=g))
    _check(pkg, img, txt, dimg, dtxt, s, s, gc=0.0, gd=1.0)


def test_output_dict_and_tuple(pkg):
    img, txt, dimg, dtxt = _inputs("clustered", 256, 128, 192, 3)
    sc, st = torch.tensor(14.29, device=DEV), torch.tensor(100.0, device=DEV)
    out = pkg.DistillClipLoss()(img, txt, sc, dimg, dtxt, st, output_dict=True)
    assert list(out) == ["contrastive_loss", "distill_loss"]
    tup = pkg.DistillClipLoss()(img, txt, sc, dimg, dtxt, st)
    assert isinstance(tup, tuple) and len(tup) == 2
    ref = distill_ref.rank_grads(img.double(), txt.double(), dimg.double(), dtxt.double(), 14.29, 100.0, 1)[0]
    for got, name in ((out["contrastive_loss"], "contrastive"), (out["distill_loss"], "distill"), (tup[0], "contrastive"),
                      (tup[1], "distill")):
        assert abs(float(got) - ref[name]) <= LOSS_RTOL * ref[name]


# ---- several ranks on one GPU through the C ABI -------------------------------------------------------------------
def _plan(lib, _cabi, b, W, r, D, Dt, row_only=False):
    h = C.c_void_p()
    flags = _cabi.DSOFT_F_DISTILL | (_cabi.DSOFT_F_ROW_ONLY if row_only else 0)
    _cabi.check(lib.dsoft_plan_create(C.byref(_cabi.Shape(b=b, world=W, rank=r, D=D, Dp=Dt, Dd=Dt, flags=flags)),
                                      C.byref(h)), "plan")
    return h


@pytest.mark.parametrize("gwg", [True, False])
@pytest.mark.parametrize("W,b,dims,ss", [(2, 520, (512, 768), (14.29, 100.0)), (4, 256, (768, 1024), (50.0, 30.0)),
                                         (8, 136, (1024, 512), (100.0, 100.0))])
def test_every_rank_through_the_abi(pkg, W, b, dims, ss, gwg):
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    D, Dt = dims
    s, st_ = ss
    B = W * b
    img, txt, dimg, dtxt = _inputs("clustered", B, D, Dt, seed=W)
    ref = distill_ref.rank_grads(img.double(), txt.double(), dimg.double(), dtxt.double(), s, st_, W,
                                 gather_with_grad=gwg, gc=GC, gd=GD)
    ls, lt = torch.tensor([s], device=DEV), torch.tensor([st_], device=DEV)
    stream = torch.cuda.current_stream().cuda_stream
    plans = [_plan(lib, _cabi, b, W, r, D, Dt, row_only=not gwg) for r in range(W)]
    gathered = torch.empty((B, 2 * D + 2 * Dt), dtype=torch.bfloat16, device=DEV)
    for r, h in enumerate(plans):  # what the all-gather of the packed rows produces
        _cabi.check(lib.dsoft_pack(h, img[r * b:].data_ptr(), _cabi.DT_F32, D, txt[r * b:].data_ptr(), _cabi.DT_F32, D,
                                   dimg[r * b:].data_ptr(), _cabi.DT_F32, Dt, dtxt[r * b:].data_ptr(), _cabi.DT_F32,
                                   Dt, gathered.data_ptr(), stream), "pack")
    states, stats, losses = [], torch.empty((W, 4, b), device=DEV), torch.empty((W, 2), device=DEV)
    for r, h in enumerate(plans):
        state = torch.empty(lib.dsoft_plan_state_bytes(h) // 4, device=DEV)
        fscr = torch.empty(lib.dsoft_plan_forward_scratch_bytes(h) // 4, device=DEV)
        _cabi.check(lib.dsoft_distill_forward(h, gathered.data_ptr(), ls.data_ptr(), lt.data_ptr(), state.data_ptr(),
                                              fscr.data_ptr(), stats[r].data_ptr(), losses[r].data_ptr(), stream),
                    "forward")
        states.append(state)
    gout = torch.tensor([GC, GD], device=DEV)
    for r, h in enumerate(plans):
        scr = torch.empty(lib.dsoft_plan_scratch_bytes(h) // 4, device=DEV)
        G = torch.empty(lib.dsoft_distill_g_bytes(h) // 2, dtype=torch.float16, device=DEV)
        d_i, d_t, d_s = torch.empty((b, D), device=DEV), torch.empty((b, D), device=DEV), torch.empty(1, device=DEV)
        stats_all = stats if gwg else stats[r]
        _cabi.check(lib.dsoft_distill_backward(h, gathered.data_ptr(), states[r].data_ptr(), scr.data_ptr(),
                                               stats_all.data_ptr(), G.data_ptr(), gout.data_ptr(), d_i.data_ptr(),
                                               d_t.data_ptr(), d_s.data_ptr(), stream), "backward")
        torch.cuda.synchronize()
        w = ref[r]
        assert abs(float(losses[r, 0]) - w["contrastive"]) <= LOSS_RTOL * abs(w["contrastive"]), r
        assert abs(float(losses[r, 1]) - w["distill"]) <= LOSS_RTOL * abs(w["distill"]), r
        assert rel_err(d_i, w["d_image"])[0] < GRAD_RTOL, r
        assert rel_err(d_t, w["d_text"])[0] < GRAD_RTOL, r
        assert abs(float(d_s) - w["d_scale"]) <= GRAD_RTOL * abs(w["d_scale"]) + 1e-6, (r, float(d_s), w["d_scale"])
    for h in plans:
        lib.dsoft_plan_destroy(h)


# ---- large batch: memory bound and sampled row blocks --------------------------------------------------------------
def test_b32768_memory_and_sampled_rows(pkg):
    B, D, Dt = 32768, 512, 768
    img, txt, dimg, dtxt = _inputs("clustered", B, D, Dt, seed=7)
    im, tx = img.clone().requires_grad_(True), txt.clone().requires_grad_(True)
    sc = torch.tensor(14.29, device=DEV, requires_grad=True)
    st = torch.tensor(100.0, device=DEV)
    mod = pkg.DistillClipLoss()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    c, d = mod(im, tx, sc, dimg, dtxt, st)
    (GC * c + GD * d).backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    # one fp16 [B x B] G, the O(B (D + Dt)) rows / operands / GEMM partials and the partial-statistics scratch
    assert peak <= 2 * B * B + 64 * B * (D + Dt), (peak, 2 * B * B)
    rows = [slice(0, 512), slice(B // 2 - 100, B // 2 + 412), slice(B - 512, B)]
    ref = distill_ref.blocked(img, txt, dimg, dtxt, 14.29, 100.0, gc=GC, gd=GD, rows=rows, cols=rows)
    assert abs(float(c) - ref["contrastive"]) <= LOSS_RTOL * ref["contrastive"]
    assert abs(float(d) - ref["distill"]) <= LOSS_RTOL * ref["distill"]
    assert abs(float(sc.grad) - ref["d_scale"]) <= GRAD_RTOL * abs(ref["d_scale"])
    for sl, want in zip(rows, ref["d_image"]):
        assert rel_err(im.grad[sl], want)[0] < GRAD_RTOL
    for sl, want in zip(rows, ref["d_text"]):
        assert rel_err(tx.grad[sl], want)[0] < GRAD_RTOL


def test_no_grad_allocates_nothing_of_size_b2(pkg):
    B, D, Dt = 8192, 512, 768
    img, txt, dimg, dtxt = _inputs("clustered", B, D, Dt, seed=9)
    sc, st = torch.tensor(14.29, device=DEV), torch.tensor(100.0, device=DEV)
    mod = pkg.DistillClipLoss()
    mod(img, txt, sc, dimg, dtxt, st)  # plan + kernel attributes once
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    with torch.no_grad():
        c, d = mod(img, txt, sc, dimg, dtxt, st)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < B * B  # a G would take 2 B^2 bytes
    ref = distill_ref.blocked(img, txt, dimg, dtxt, 14.29, 100.0)
    assert abs(float(c) - ref["contrastive"]) <= LOSS_RTOL * ref["contrastive"]
    assert abs(float(d) - ref["distill"]) <= LOSS_RTOL * ref["distill"]


def test_graph_capture_replays_eager_values(pkg):
    B, D, Dt = 2048, 512, 768
    img, txt, dimg, dtxt = _inputs("aligned", B, D, Dt, seed=11)
    leaves = [img.clone().requires_grad_(True), txt.clone().requires_grad_(True),
              torch.tensor(14.29, device=DEV, requires_grad=True)]
    st = torch.tensor(100.0, device=DEV)
    mod = pkg.DistillClipLoss()

    def step():
        for t in leaves:
            t.grad = None
        c, d = mod(leaves[0], leaves[1], leaves[2], dimg, dtxt, st)
        (GC * c + GD * d).backward()
        return c, d

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):  # the warm-up of the capture below
            want = [float(x) for x in step()]
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    want_g = [t.grad.clone() for t in leaves]
    for t in leaves:
        t.grad = None
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        c, d = mod(leaves[0], leaves[1], leaves[2], dimg, dtxt, st)
        (GC * c + GD * d).backward()
    g.replay()
    torch.cuda.synchronize()
    assert [float(c), float(d)] == want
    for t, w in zip(leaves, want_g):
        assert torch.equal(t.grad, w)


def test_errors(pkg):
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    img, txt, dimg, dtxt = _inputs("clustered", 64, 64, 96, 1)
    sc, st = torch.tensor(10.0, device=DEV), torch.tensor(100.0, device=DEV)
    with pytest.raises(ValueError):
        pkg.DistillClipLoss()(img, txt[:32], sc, dimg, dtxt, st)
    with pytest.raises(ValueError):
        pkg.DistillClipLoss()(img, txt, sc, dimg, dtxt[:, :64], st)
    with pytest.raises(ValueError, match="teacher"):
        pkg.DistillClipLoss()(img, txt, sc, dimg.clone().requires_grad_(True), dtxt, st)
    with pytest.raises(RuntimeError):
        pkg.DistillClipLoss()(img, txt.cpu(), sc, dimg, dtxt, st)
    # the DINO-Soft and SigLIP entry points refuse a distill plan, the distill ones refuse other plans
    h = _plan(lib, _cabi, 64, 1, 0, 64, 96)
    gathered = torch.zeros((64, 2 * 64 + 2 * 96), dtype=torch.bfloat16, device=DEV)
    buf = torch.zeros(1 << 20, device=DEV)
    lam = (C.c_float * 4)(1, 0, 0, 0)
    p = buf.data_ptr()
    assert lib.dsoft_forward(h, gathered.data_ptr(), p, lam, p, p, p, p, None, None) == EINVAL
    assert b"dsoft_distill_forward" in lib.dsoft_last_error()
    assert lib.dsoft_backward(h, gathered.data_ptr(), p, p, p, p, lam, p, p, None, p, None) == EINVAL
    assert lib.dsoft_siglip_forward(h, gathered.data_ptr(), p, None, p, p, None, p, None) == EINVAL
    assert lib.dsoft_distill_backward(h, gathered.data_ptr(), p, p, p, p + 2, p, p, p, p, None) == EINVAL  # misaligned
    lib.dsoft_plan_destroy(h)
    h2 = C.c_void_p()
    _cabi.check(lib.dsoft_plan_create(C.byref(_cabi.Shape(b=64, world=1, rank=0, D=64)), C.byref(h2)), "plan")
    assert lib.dsoft_distill_g_bytes(h2) == 0
    assert lib.dsoft_distill_forward(h2, gathered.data_ptr(), p, p, p, p, p, p, None) == EINVAL
    lib.dsoft_plan_destroy(h2)


# ---- two GPUs, NCCL ------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, B, D, Dt, gwg, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import dinosoft_b200 as pkg

    img, txt, _ = synth(5, B, D, 8)
    dimg, dtxt, _ = synth(6, B, Dt, 8)
    b = B // world
    dev = torch.device("cuda", rank)
    sl = slice(rank * b, (rank + 1) * b)
    im = img[sl].to(dev).requires_grad_(True)
    tx = txt[sl].to(dev).requires_grad_(True)
    sc = torch.tensor(14.29, device=dev, requires_grad=True)
    mod = pkg.DistillClipLoss(local_loss=True, gather_with_grad=gwg, rank=rank, world_size=world)
    c, d = mod(im, tx, sc, dimg[sl].to(dev), dtxt[sl].to(dev), torch.tensor(100.0, device=dev))
    (GC * c + GD * d).backward()
    torch.cuda.synchronize()
    ret[rank] = dict(contrastive=float(c.detach()), distill=float(d.detach()), d_image=im.grad.cpu(),
                     d_text=tx.grad.cpu(), d_scale=float(sc.grad))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("gwg", [True, False])
def test_two_gpus_nccl(gwg):
    B, D, Dt, world = 2048, 512, 768, 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), B, D, Dt, gwg, ret), nprocs=world, join=True)
    img, txt, _ = synth(5, B, D, 8)
    dimg, dtxt, _ = synth(6, B, Dt, 8)
    ref = distill_ref.rank_grads(img, txt, dimg, dtxt, 14.29, 100.0, world, gather_with_grad=gwg, gc=GC, gd=GD)
    for r in range(world):
        o, w = ret[r], ref[r]
        for k in ("contrastive", "distill"):
            assert abs(o[k] - w[k]) <= LOSS_RTOL * abs(w[k])
        assert rel_err(o["d_image"], w["d_image"])[0] < GRAD_RTOL
        assert rel_err(o["d_text"], w["d_text"])[0] < GRAD_RTOL
        assert abs(o["d_scale"] - w["d_scale"]) <= GRAD_RTOL * abs(w["d_scale"]) + 1e-6
