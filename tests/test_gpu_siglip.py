"""SigLipLoss on the B200 (siglip.py -> dsoft_siglip_forward / _backward -> dsoft_fwd_kernel<MODE_SIGLIP> + the
gradient GEMMs) against the fp64 statement of upstream's recipe (tests/siglip_ref.py).

Bars: loss 1e-4 relative; d_image / d_text 1e-3 (max error over max magnitude; a bf16 gradient may in addition be off
by its own rounding, 2^-8 of the element - the module returns gradients in the input dtype); d_scale / d_bias 1e-3
relative.  Inputs are bf16-representable, so kernel and statement see the same operands."""
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
import siglip_ref

pytestmark = pytest.mark.gpu

LOSS_RTOL, GRAD_RTOL = 1e-4, 1e-3
DEV = "cuda"
EINVAL = -1


def _inputs(kind, B, D, seed):
    if kind == "aligned":
        img, txt, _ = synth_aligned(seed, B, D, 8)
    else:
        img, txt, _ = synth(seed, B, D, 8, clustered=(kind == "clustered"))
    return img.to(DEV), txt.to(DEV)


def _scalar_ok(got, want, scale_abs):
    return abs(got - want) <= GRAD_RTOL * abs(want) + 1e-6 * scale_abs


def _check(pkg, img, txt, s, beta, dtype=torch.float32, noncontig=False):
    ref = siglip_ref.rank_grads(img.double(), txt.double(), s, beta, 1)[0]
    im, tx = img.to(dtype), txt.to(dtype)
    if noncontig:  # every other column of a wider buffer
        wide_i = torch.zeros((im.shape[0], 2 * im.shape[1]), dtype=dtype, device=DEV)
        wide_t = torch.zeros_like(wide_i)
        wide_i[:, ::2], wide_t[:, ::2] = im, tx
        im, tx = wide_i[:, ::2], wide_t[:, ::2]
        assert not im.is_contiguous()
    im, tx = im.detach().requires_grad_(True), tx.detach().requires_grad_(True)
    sc = torch.tensor(float(s), device=DEV, requires_grad=True)
    bi = None if beta is None else torch.tensor(float(beta), device=DEV, requires_grad=True)
    loss = pkg.SigLipLoss()(im, tx, sc, bi)
    loss.backward()
    torch.cuda.synchronize()
    assert loss.shape == () and loss.dtype == torch.float32
    assert im.grad.dtype == dtype and tx.grad.dtype == dtype
    assert abs(float(loss) - ref["loss"]) <= LOSS_RTOL * abs(ref["loss"]), (float(loss), ref["loss"])
    out_round = 2.0 ** -8 if dtype == torch.bfloat16 else 0.0
    for name, got, want in (("d_image", im.grad, ref["d_image"]), ("d_text", tx.grad, ref["d_text"])):
        excess = (got.double() - want).abs() - out_round * want.abs()
        err = excess.max().item() / want.abs().max().item()
        assert err < GRAD_RTOL, (name, err)
    # absolute scale of the scalar gradients: the sums of |terms|
    x = img.double() @ txt.double().T
    absg = torch.sigmoid(-(s * x + (beta or 0.0)).abs()).sum().item() + img.shape[0]
    assert _scalar_ok(float(sc.grad), ref["d_scale"], absg / img.shape[0]), (float(sc.grad), ref["d_scale"])
    if beta is not None:
        assert _scalar_ok(float(bi.grad), ref["d_bias"], absg / img.shape[0]), (float(bi.grad), ref["d_bias"])
    return loss


CASES = [  # B, D, (s, beta), input kind, dtype, non-contiguous
    (1, 512, (10.0, -10.0), "clustered", torch.float32, False),
    (7, 64, (10.0, -10.0), "aligned", torch.float32, False),
    (130, 100, (100.0, 0.0), "random", torch.float32, False),  # D padded to 104
    (300, 512, (30.0, -5.0), "clustered", torch.bfloat16, False),
    (1000, 768, (10.0, -10.0), "aligned", torch.float16, False),
    (1000, 768, (10.0, None), "clustered", torch.float32, True),
    (2049, 1024, (100.0, 0.0), "aligned", torch.bfloat16, False),
    (4133, 512, (30.0, -5.0), "random", torch.float16, True),
    (8192, 512, (10.0, -10.0), "aligned", torch.float32, False),
    (8192, 768, (100.0, None), "clustered", torch.bfloat16, False),
    (8192, 1024, (30.0, -5.0), "clustered", torch.float32, False),
]


@pytest.mark.parametrize("B,D,sb,kind,dtype,noncontig", CASES)
def test_module_against_fp64(pkg, B, D, sb, kind, dtype, noncontig):
    img, txt = _inputs(kind, B, D, seed=B + D)
    _check(pkg, img, txt, sb[0], sb[1], dtype, noncontig)


def test_output_dict_and_no_bias_gradient(pkg):
    img, txt = _inputs("clustered", 256, 128, 3)
    out = pkg.SigLipLoss()(img, txt, torch.tensor(10.0, device=DEV), torch.tensor(-10.0, device=DEV), output_dict=True)
    assert list(out) == ["contrastive_loss"]
    ref = siglip_ref.rank_grads(img.double(), txt.double(), 10.0, -10.0, 1)[0]
    assert abs(float(out["contrastive_loss"]) - ref["loss"]) <= LOSS_RTOL * ref["loss"]


# ---- several ranks on one GPU through the C ABI -------------------------------------------------------------------
def _plan(lib, _cabi, b, W, r, D):
    h = C.c_void_p()
    _cabi.check(lib.dsoft_plan_create(C.byref(_cabi.Shape(b=b, world=W, rank=r, D=D, flags=_cabi.DSOFT_F_SIGLIP)),
                                      C.byref(h)), "plan")
    return h


@pytest.mark.parametrize("W,b,D,sb", [(2, 520, 512, (10.0, -10.0)), (4, 256, 768, (30.0, -5.0)),
                                      (8, 136, 1024, (100.0, None))])
def test_every_rank_through_the_abi(pkg, W, b, D, sb):
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    s, beta = sb
    B = W * b
    img, txt = _inputs("clustered", B, D, seed=W)
    ref = siglip_ref.rank_grads(img.double(), txt.double(), s, beta, W)
    ls = torch.tensor([s], device=DEV)
    lb = None if beta is None else torch.tensor([beta], device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    plans = [_plan(lib, _cabi, b, W, r, D) for r in range(W)]
    gathered = torch.empty((B, 2 * D), dtype=torch.bfloat16, device=DEV)
    for r, h in enumerate(plans):  # what the all-gather of the packed rows produces
        _cabi.check(lib.dsoft_pack(h, img[r * b:].data_ptr(), _cabi.DT_F32, D, txt[r * b:].data_ptr(), _cabi.DT_F32, D,
                                   None, 0, 0, None, 0, 0, gathered.data_ptr(), st), "pack")
    ptr = lambda t: None if t is None else t.data_ptr()
    for r, h in enumerate(plans):
        state = torch.empty(lib.dsoft_plan_state_bytes(h) // 4, device=DEV)
        fscr = torch.empty(lib.dsoft_plan_forward_scratch_bytes(h) // 4, device=DEV)
        scr = torch.empty(lib.dsoft_plan_scratch_bytes(h) // 4, device=DEV)
        G = torch.empty(lib.dsoft_siglip_g_bytes(h) // 2, dtype=torch.float16, device=DEV)
        loss = torch.empty(1, device=DEV)
        _cabi.check(lib.dsoft_siglip_forward(h, gathered.data_ptr(), ls.data_ptr(), ptr(lb), state.data_ptr(),
                                             fscr.data_ptr(), G.data_ptr(), loss.data_ptr(), st), "forward")
        gout = torch.tensor([0.75], device=DEV)
        d_i, d_t = torch.empty((b, D), device=DEV), torch.empty((b, D), device=DEV)
        d_s, d_b = torch.empty(1, device=DEV), torch.empty(1, device=DEV)
        _cabi.check(lib.dsoft_siglip_backward(h, gathered.data_ptr(), state.data_ptr(), scr.data_ptr(), G.data_ptr(),
                                              gout.data_ptr(), d_i.data_ptr(), d_t.data_ptr(), d_s.data_ptr(),
                                              d_b.data_ptr(), st), "backward")
        torch.cuda.synchronize()
        w = ref[r]
        assert abs(float(loss) - w["loss"]) <= LOSS_RTOL * abs(w["loss"]), (r, float(loss), w["loss"])
        assert rel_err(d_i, 0.75 * w["d_image"])[0] < GRAD_RTOL, r
        assert rel_err(d_t, 0.75 * w["d_text"])[0] < GRAD_RTOL, r
        assert abs(float(d_s) - 0.75 * w["d_scale"]) <= GRAD_RTOL * abs(0.75 * w["d_scale"]) + 1e-6, r
        if beta is not None:
            assert abs(float(d_b) - 0.75 * w["d_bias"]) <= GRAD_RTOL * abs(0.75 * w["d_bias"]) + 1e-6, r
    for h in plans:
        lib.dsoft_plan_destroy(h)


# ---- large batch: memory bound and sampled row blocks --------------------------------------------------------------
def test_b32768_memory_and_sampled_rows(pkg):
    B, D = 32768, 768
    img, txt = _inputs("clustered", B, D, seed=7)
    im, tx = img.clone().requires_grad_(True), txt.clone().requires_grad_(True)
    sc = torch.tensor(10.0, device=DEV, requires_grad=True)
    bi = torch.tensor(-10.0, device=DEV, requires_grad=True)
    mod = pkg.SigLipLoss()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    loss = mod(im, tx, sc, bi)
    loss.backward()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak <= 2 * B * B + 64 * B * D, (peak, 2 * B * B)
    rows = [slice(0, 512), slice(B // 2 - 100, B // 2 + 412), slice(B - 512, B)]
    ref = siglip_ref.blocked(img, txt, 10.0, -10.0, rows=rows, cols=rows)
    assert abs(float(loss) - ref["loss"]) <= LOSS_RTOL * ref["loss"]
    assert abs(float(sc.grad) - ref["d_scale"]) <= GRAD_RTOL * abs(ref["d_scale"])
    assert abs(float(bi.grad) - ref["d_bias"]) <= GRAD_RTOL * abs(ref["d_bias"])
    for sl, want in zip(rows, ref["d_image"]):
        assert rel_err(im.grad[sl], want)[0] < GRAD_RTOL
    for sl, want in zip(rows, ref["d_text"]):
        assert rel_err(tx.grad[sl], want)[0] < GRAD_RTOL


def test_forward_without_gradient_allocates_no_g(pkg):
    B, D = 8192, 512
    img, txt = _inputs("clustered", B, D, seed=9)
    sc, bi = torch.tensor(10.0, device=DEV), torch.tensor(-10.0, device=DEV)
    mod = pkg.SigLipLoss()
    mod(img, txt, sc, bi)  # plan + kernel attributes once
    for ctx, args in ((torch.no_grad(), (img, txt)), (torch.enable_grad(), (img, txt))):  # nothing requires grad
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        with ctx:
            loss = mod(*args, sc, bi)
        torch.cuda.synchronize()
        assert torch.cuda.max_memory_allocated() - base < B * B  # a G would take 2 B^2 bytes
        ref = siglip_ref.blocked(img, txt, 10.0, -10.0)
        assert abs(float(loss) - ref["loss"]) <= LOSS_RTOL * ref["loss"]


def _step(pkg, mod, im, tx, sc, bi):
    for t in (im, tx, sc, bi):
        t.grad = None
    loss = mod(im, tx, sc, bi)
    loss.backward()
    return loss


def test_side_stream_and_graph_capture(pkg):
    B, D = 2048, 512
    img, txt = _inputs("aligned", B, D, seed=11)
    leaves = [img.clone().requires_grad_(True), txt.clone().requires_grad_(True),
              torch.tensor(10.0, device=DEV, requires_grad=True), torch.tensor(-10.0, device=DEV, requires_grad=True)]
    mod = pkg.SigLipLoss()
    want_loss = float(_step(pkg, mod, *leaves))
    want = [t.grad.clone() for t in leaves]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):  # also the warm-up of the capture below
            loss = _step(pkg, mod, *leaves)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    assert float(loss) == want_loss
    for t, w in zip(leaves, want):
        assert torch.equal(t.grad, w)
    for t in leaves:
        t.grad = None
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        loss = mod(*leaves)
        loss.backward()
    with torch.no_grad():  # new inputs in the captured buffers
        leaves[0].copy_(txt)
        leaves[1].copy_(img)
    g.replay()
    torch.cuda.synchronize()
    ref = siglip_ref.rank_grads(txt.double(), img.double(), 10.0, -10.0, 1)[0]
    assert abs(float(loss) - ref["loss"]) <= LOSS_RTOL * ref["loss"]
    assert rel_err(leaves[0].grad, ref["d_image"])[0] < GRAD_RTOL
    assert rel_err(leaves[1].grad, ref["d_text"])[0] < GRAD_RTOL


def test_errors(pkg):
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    img, txt = _inputs("clustered", 64, 64, 1)
    sc = torch.tensor(10.0, device=DEV)
    with pytest.raises(ValueError):
        pkg.SigLipLoss()(img, txt[:32], sc)
    with pytest.raises(ValueError):
        pkg.SigLipLoss()(img[0], txt[0], sc)
    with pytest.raises(RuntimeError):
        pkg.SigLipLoss()(img, txt.cpu(), sc)
    # the DINO-Soft entry points refuse a SigLIP plan, the SigLIP ones refuse a DINO-Soft plan
    h = _plan(lib, _cabi, 64, 1, 0, 64)
    gathered = torch.zeros((64, 128), dtype=torch.bfloat16, device=DEV)
    buf = torch.zeros(1 << 20, device=DEV)
    lam = (C.c_float * 4)(1, 0, 0, 0)
    p = buf.data_ptr()
    assert lib.dsoft_forward(h, gathered.data_ptr(), p, lam, p, p, p, p, None, None) == EINVAL
    assert b"dsoft_siglip_forward" in lib.dsoft_last_error()
    assert lib.dsoft_backward(h, gathered.data_ptr(), p, p, p, p, lam, p, p, None, p, None) == EINVAL
    assert lib.dsoft_siglip_forward(h, gathered.data_ptr(), p, None, p, p, p + 2, p, None) == EINVAL  # misaligned G
    lib.dsoft_plan_destroy(h)
    h2 = C.c_void_p()
    _cabi.check(lib.dsoft_plan_create(C.byref(_cabi.Shape(b=64, world=1, rank=0, D=64)), C.byref(h2)), "plan")
    assert lib.dsoft_siglip_g_bytes(h2) == 0
    assert lib.dsoft_siglip_forward(h2, gathered.data_ptr(), p, None, p, p, None, p, None) == EINVAL
    lib.dsoft_plan_destroy(h2)


# ---- two GPUs, NCCL ------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, B, D, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import dinosoft_b200 as pkg

    img, txt, _ = synth(5, B, D, 8)
    b = B // world
    dev = torch.device("cuda", rank)
    im = img[rank * b:(rank + 1) * b].to(dev).requires_grad_(True)
    tx = txt[rank * b:(rank + 1) * b].to(dev).requires_grad_(True)
    sc = torch.tensor(10.0, device=dev, requires_grad=True)
    bi = torch.tensor(-10.0, device=dev, requires_grad=True)
    loss = pkg.SigLipLoss(rank=rank, world_size=world, dist_impl="gather")(im, tx, sc, bi)
    loss.backward()
    torch.cuda.synchronize()
    ret[rank] = dict(loss=float(loss.detach()), d_image=im.grad.cpu(), d_text=tx.grad.cpu(), d_scale=float(sc.grad),
                     d_bias=float(bi.grad))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_nccl():
    B, D, world = 2048, 512, 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), B, D, ret), nprocs=world, join=True)
    img, txt, _ = synth(5, B, D, 8)
    ref = siglip_ref.rank_grads(img, txt, 10.0, -10.0, world)
    for r in range(world):
        o, w = ret[r], ref[r]
        assert abs(o["loss"] - w["loss"]) <= LOSS_RTOL * abs(w["loss"])
        assert rel_err(o["d_image"], w["d_image"])[0] < GRAD_RTOL
        assert rel_err(o["d_text"], w["d_text"])[0] < GRAD_RTOL
        assert abs(o["d_scale"] - w["d_scale"]) <= GRAD_RTOL * abs(w["d_scale"]) + 1e-6
        assert abs(o["d_bias"] - w["d_bias"]) <= GRAD_RTOL * abs(w["d_bias"]) + 1e-6
