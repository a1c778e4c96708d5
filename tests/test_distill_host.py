"""DistillClipLoss (distill.py, dsoft_distill_*) on the CPU: the C-ABI surface, plan validation, the module's signatures
and error paths against upstream, install / uninstall into a fake open_clip, and the fp64 statement
(tests/distill_ref.py) against upstream's `gather_features` + `DistillClipLoss.forward` run as a real gloo job."""
import ctypes as C
import inspect
import os
import re
import socket
import sys
import types

import pytest
import torch
import torch.distributed as dist
import torch.distributed.nn  # noqa: F401  (all_gather with gradient)
import torch.multiprocessing as mp

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tests"))
import distill_ref  # noqa: E402

REF_LOSS = os.path.join(ROOT, "oracle", "_ref", "loss.py")


def _header():
    return re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dsoft.h")).read(), flags=re.S)


def test_abi_table_matches_header(pkg):
    from dinosoft_b200 import _cabi

    text = _header()
    for name in ("dsoft_distill_g_bytes", "dsoft_distill_forward", "dsoft_distill_backward"):
        m = re.search(rf"\b{name}\s*\(([^)]*)\)", text)
        assert m, name
        nargs = len([a for a in m.group(1).split(",") if a.strip()])
        assert len(_cabi.PROTOTYPES[name][1]) == nargs, name
    raw = open(os.path.join(ROOT, "include", "dsoft.h")).read()
    assert int(re.search(r"#define DSOFT_F_DISTILL (\d+)u", raw).group(1)) == _cabi.DSOFT_F_DISTILL
    # the distill calls were added to 0.2.6 without a version change: header and library agree on it
    version = int(re.search(r"#define DSOFT_VERSION (\d+)", raw).group(1))
    assert version >= 260 and _cabi.lib().dsoft_version() == version


@pytest.mark.parametrize("bad", [dict(Dp=0), dict(Dp=64), dict(Dd=0, Dp=0), dict(flags=256 | 1, teacher_temp=0.1),
                                 dict(flags=256 | 2), dict(flags=256 | 16), dict(flags=256 | 32, c_clip=1.0),
                                 dict(flags=256 | 128), dict(flags=256 | 8), dict(flags=256 | 4, world=2, b=64)])
def test_distill_plan_rejects_other_terms(pkg, bad):
    """Checked before any device query, so also without a GPU.  DSOFT_F_ROW_ONLY only at world > 1."""
    from dinosoft_b200 import _cabi

    kw = dict(b=128, world=1, rank=0, D=64, Dp=96, Dd=96, flags=_cabi.DSOFT_F_DISTILL)
    kw.update(bad)
    h = C.c_void_p()
    assert _cabi.lib().dsoft_plan_create(C.byref(_cabi.Shape(**kw)), C.byref(h)) == -1
    assert b"DSOFT_F_" in _cabi.lib().dsoft_last_error()
    if not kw["flags"] & (1 | 2 | 32 | 128):  # the other terms' own checks may speak first; these are ours
        assert b"DSOFT_F_DISTILL" in _cabi.lib().dsoft_last_error()


def test_null_plan_calls_fail(pkg):
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    assert lib.dsoft_distill_g_bytes(None) == 0
    assert lib.dsoft_distill_forward(*([None] * 9)) == -1
    assert lib.dsoft_distill_backward(*([None] * 11)) == -1


UPSTREAM_INIT = ["self", "local_loss", "gather_with_grad", "cache_labels", "rank", "world_size", "use_horovod"]
UPSTREAM_FORWARD = ["self", "image_features", "text_features", "logit_scale", "dist_image_features",
                    "dist_text_features", "dist_logit_scale", "output_dict"]


def test_signatures_match_upstream(pkg):
    init = inspect.signature(pkg.DistillClipLoss.__init__).parameters
    assert list(init) == UPSTREAM_INIT + ["process_group"]
    assert [init[k].default for k in UPSTREAM_INIT[1:]] == [False, False, False, 0, 1, False]
    assert init["process_group"].default is None
    fwd = inspect.signature(pkg.DistillClipLoss.forward).parameters
    assert list(fwd) == UPSTREAM_FORWARD
    assert fwd["output_dict"].default is False
    if os.path.exists(REF_LOSS):
        ref = _ref_module()
        if hasattr(ref, "DistillClipLoss"):
            assert list(inspect.signature(ref.DistillClipLoss.__init__).parameters) == UPSTREAM_INIT
            assert list(inspect.signature(ref.DistillClipLoss.forward).parameters) == UPSTREAM_FORWARD


def _cpu_args(b=4, D=8, Dt=12, teacher_grad=False):
    x = torch.randn(b, D)
    t = torch.randn(b, Dt, requires_grad=teacher_grad)
    return x, x.clone(), torch.tensor(10.0), t, torch.randn(b, Dt), torch.tensor(100.0)


def test_error_paths(pkg):
    M = pkg.DistillClipLoss
    with pytest.raises(RuntimeError, match="CUDA"):
        M()(*_cpu_args())
    a = list(_cpu_args())
    a[1] = torch.randn(5, 8)
    with pytest.raises(ValueError):
        M()(*a)
    a = list(_cpu_args())
    a[4] = torch.randn(4, 16)
    with pytest.raises(ValueError):
        M()(*a)
    a = list(_cpu_args())
    a[3] = torch.randn(3, 12)
    a[4] = torch.randn(3, 12)
    with pytest.raises(ValueError):
        M()(*a)
    with pytest.raises(ValueError, match="teacher"):
        M()(*_cpu_args(teacher_grad=True))
    with torch.no_grad():  # a teacher leaf that requires grad is fine while grad is off: nothing flows back
        with pytest.raises(RuntimeError, match="CUDA"):
            M()(*_cpu_args(teacher_grad=True))
    with pytest.raises(NotImplementedError, match="Horovod"):
        M(use_horovod=True)(*_cpu_args())
    with pytest.raises(NotImplementedError, match="--local-loss"):
        M(rank=0, world_size=2)(*_cpu_args())


def _fake_open_clip():
    class Clip:  # stand-ins for the fork's classes
        pass

    class Dcl:
        pass

    loss = types.ModuleType("open_clip.loss")
    factory = types.ModuleType("open_clip.factory")
    train = types.ModuleType("open_clip_train.train")
    for m in (loss, factory):
        m.ClipLossWithDINOEnhancements, m.DistillClipLoss = Clip, Dcl
    train.DistillClipLoss = Dcl
    return types.SimpleNamespace(loss=loss, factory=factory), train, Dcl


def test_install_and_uninstall(pkg, monkeypatch):
    oc, train, Dcl = _fake_open_clip()
    monkeypatch.setitem(sys.modules, "open_clip_train.train", train)
    pkg.install_into_open_clip(oc)  # default: the distill loss stays upstream's
    assert oc.loss.DistillClipLoss is Dcl and oc.factory.DistillClipLoss is Dcl and train.DistillClipLoss is Dcl
    assert not hasattr(oc.loss, "_reference_DistillClipLoss")
    pkg.install_into_open_clip(oc, distill=True)
    assert oc.loss.DistillClipLoss is pkg.DistillClipLoss and oc.factory.DistillClipLoss is pkg.DistillClipLoss
    assert train.DistillClipLoss is pkg.DistillClipLoss
    pkg.install_into_open_clip(oc, distill=True)  # twice: the saved original is kept
    assert oc.loss._reference_DistillClipLoss is Dcl
    pkg.uninstall_from_open_clip(oc)
    assert oc.loss.DistillClipLoss is Dcl and oc.factory.DistillClipLoss is Dcl and train.DistillClipLoss is Dcl


# ---- the fp64 statement against the upstream recipe ---------------------------------------------------------------
def _inputs(B, D, Dt, seed=0):
    g = torch.Generator().manual_seed(seed)
    n = torch.nn.functional.normalize
    img = n(torch.randn(B, D, generator=g, dtype=torch.float64), dim=-1)
    txt = n(img + 0.7 * torch.randn(B, D, generator=g, dtype=torch.float64), dim=-1)
    dimg = n(torch.randn(B, Dt, generator=g, dtype=torch.float64), dim=-1)
    dtxt = n(dimg + 0.5 * torch.randn(B, Dt, generator=g, dtype=torch.float64), dim=-1)
    return img, txt, dimg, dtxt


S, ST, GC, GD = 14.0, 30.0, 0.3, 1.7


def test_statement_world1_is_the_plain_recipe():
    img, txt, dimg, dtxt = _inputs(37, 16, 24)
    x, t = S * img @ txt.T, ST * dimg @ dtxt.T
    lab = torch.arange(37)
    ce = torch.nn.functional.cross_entropy
    want_c = (ce(x, lab) + ce(x.T, lab)) / 2
    kl = lambda tt, ss: -(tt.softmax(1) * ss.log_softmax(1)).sum(1).mean(0)  # noqa: E731
    want_d = (kl(t, x) + kl(t.T, x.T)) / 2
    full = distill_ref.rank_grads(img, txt, dimg, dtxt, S, ST, 1, gc=GC, gd=GD)[0]
    assert full["contrastive"] == pytest.approx(float(want_c), rel=1e-14)
    assert full["distill"] == pytest.approx(float(want_d), rel=1e-14)
    blk = distill_ref.blocked(img, txt, dimg, dtxt, S, ST, gc=GC, gd=GD, rows=[slice(0, 37)], cols=[slice(5, 20)],
                              block=8)
    assert blk["contrastive"] == pytest.approx(full["contrastive"], rel=1e-12)
    assert blk["distill"] == pytest.approx(full["distill"], rel=1e-12)
    assert blk["d_scale"] == pytest.approx(full["d_scale"], rel=1e-12)
    assert torch.allclose(blk["d_image"][0], full["d_image"], rtol=1e-12, atol=1e-15)
    assert torch.allclose(blk["d_text"][0], full["d_text"][5:20], rtol=1e-12, atol=1e-15)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _ref_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("dsoft_ref_loss_distill", REF_LOSS)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _gather_features(image_features, text_features, gather_with_grad, rank, world):
    """Upstream gather_features with local_loss=True, restated."""
    if gather_with_grad:
        return (torch.cat(torch.distributed.nn.all_gather(image_features), dim=0),
                torch.cat(torch.distributed.nn.all_gather(text_features), dim=0))
    gi = [torch.zeros_like(image_features) for _ in range(world)]
    gt = [torch.zeros_like(text_features) for _ in range(world)]
    dist.all_gather(gi, image_features)
    dist.all_gather(gt, text_features)
    return torch.cat(gi, dim=0), torch.cat(gt, dim=0)


def _upstream_forward(im, tx, sc, dim, dtx, dsc, gather_with_grad, rank, world):
    """Upstream DistillClipLoss.forward (ClipLoss.get_logits with local_loss, then the CE / dist_loss), restated."""
    all_i, all_t = _gather_features(im, tx, gather_with_grad, rank, world)
    all_di, all_dt = _gather_features(dim, dtx, gather_with_grad, rank, world)
    lpi, lpt = sc * im @ all_t.T, sc * tx @ all_i.T
    dpi, dpt = dsc * dim @ all_dt.T, dsc * dtx @ all_di.T
    labels = torch.arange(im.shape[0]) + rank * im.shape[0]
    ce = torch.nn.functional.cross_entropy
    contrastive = (ce(lpi, labels) + ce(lpt, labels)) / 2
    kl = lambda tt, ss: -(tt.softmax(dim=1) * ss.log_softmax(dim=1)).sum(dim=1).mean(dim=0)  # noqa: E731
    distill = (kl(dpi, lpi) + kl(dpt, lpt)) / 2
    return contrastive, distill


def _worker(rank, world, port, B, D, Dt, use_ref, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    img, txt, dimg, dtxt = _inputs(B, D, Dt)
    b = B // world
    sl = slice(rank * b, (rank + 1) * b)
    ref = _ref_module() if use_ref else None
    out = {}
    for gwg in (True, False):
        im = img[sl].clone().requires_grad_(True)
        tx = txt[sl].clone().requires_grad_(True)
        sc = torch.tensor(S, dtype=torch.float64, requires_grad=True)
        dsc = torch.tensor(ST, dtype=torch.float64)
        if ref is None:
            c, d = _upstream_forward(im, tx, sc, dimg[sl], dtxt[sl], dsc, gwg, rank, world)
        else:
            c, d = ref.DistillClipLoss(local_loss=True, gather_with_grad=gwg, rank=rank, world_size=world)(
                im, tx, sc, dimg[sl], dtxt[sl], dsc)
        (GC * c + GD * d).backward()
        out[gwg] = dict(contrastive=float(c.detach()), distill=float(d.detach()), d_image=im.grad.clone(),
                        d_text=tx.grad.clone(), d_scale=float(sc.grad))
    ret[rank] = out
    dist.barrier()
    dist.destroy_process_group()


def _check(outs, B, D, Dt, world):
    img, txt, dimg, dtxt = _inputs(B, D, Dt)
    for gwg in (True, False):
        want = distill_ref.rank_grads(img, txt, dimg, dtxt, S, ST, world, gather_with_grad=gwg, gc=GC, gd=GD)
        for r, per in enumerate(outs):
            o, w = per[gwg], want[r]
            for k in ("contrastive", "distill"):
                assert o[k] == pytest.approx(w[k], rel=1e-12, abs=1e-12), (r, gwg, k)
            assert o["d_scale"] == pytest.approx(w["d_scale"], rel=1e-10, abs=1e-10), (r, gwg)
            for k in ("d_image", "d_text"):
                assert torch.allclose(o[k], w[k], rtol=1e-10, atol=1e-10), (r, gwg, k)


def _spawn(world, B, D, Dt, use_ref):
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), B, D, Dt, use_ref, ret), nprocs=world, join=True)
    return [ret[r] for r in range(world)]


@pytest.mark.parametrize("world", [2, 3])
def test_statement_matches_upstream_recipe_gloo(world):
    """Per-rank losses and gradients of upstream's recipe under gloo, gather_with_grad on and off."""
    B, D, Dt = 10 * world, 16, 24
    _check(_spawn(world, B, D, Dt, False), B, D, Dt, world)


@pytest.mark.skipif(not os.path.exists(REF_LOSS), reason="oracle/_ref/loss.py is not staged")
def test_statement_matches_staged_reference():
    if not hasattr(_ref_module(), "DistillClipLoss"):
        pytest.skip("the staged reference has no DistillClipLoss")
    B, D, Dt, world = 20, 16, 24, 2
    _check(_spawn(world, B, D, Dt, True), B, D, Dt, world)
