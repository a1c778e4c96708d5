"""SigLipLoss (siglip.py, dsoft_siglip_*) on the CPU: the C-ABI surface, plan validation, the module's signatures and
dist_impl check against upstream, install / uninstall into a fake open_clip, and the fp64 statement
(tests/siglip_ref.py) against the upstream `gather` recipe run as a real gloo job."""
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
import siglip_ref  # noqa: E402

REF_LOSS = os.path.join(ROOT, "oracle", "_ref", "loss.py")


def _header():
    return re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dsoft.h")).read(), flags=re.S)


def test_abi_table_matches_header(pkg):
    from dinosoft_b200 import _cabi

    text = _header()
    for name in ("dsoft_siglip_g_bytes", "dsoft_siglip_forward", "dsoft_siglip_backward"):
        m = re.search(rf"\b{name}\s*\(([^)]*)\)", text)
        assert m, name
        nargs = len([a for a in m.group(1).split(",") if a.strip()])
        assert len(_cabi.PROTOTYPES[name][1]) == nargs, name
    raw = open(os.path.join(ROOT, "include", "dsoft.h")).read()
    assert int(re.search(r"#define DSOFT_F_SIGLIP (\d+)u", raw).group(1)) == _cabi.DSOFT_F_SIGLIP
    assert int(re.search(r"#define DSOFT_VERSION (\d+)", raw).group(1)) == 260
    assert _cabi.lib().dsoft_version() == 260


@pytest.mark.parametrize("bad", [dict(Dd=64), dict(Dp=64), dict(flags=1 | 128, Dd=64, teacher_temp=0.1),
                                 dict(flags=128 | 16), dict(flags=128 | 8, world=2, b=64)])
def test_siglip_plan_rejects_other_terms(pkg, bad):
    """Checked before any device query, so also without a GPU."""
    from dinosoft_b200 import _cabi

    kw = dict(b=128, world=1, rank=0, D=64, Dp=0, Dd=0, flags=_cabi.DSOFT_F_SIGLIP)
    kw.update(bad)
    h = C.c_void_p()
    assert _cabi.lib().dsoft_plan_create(C.byref(_cabi.Shape(**kw)), C.byref(h)) == -1
    assert b"DSOFT_F_SIGLIP" in _cabi.lib().dsoft_last_error()


def test_null_plan_calls_fail(pkg):
    from dinosoft_b200 import _cabi

    lib = _cabi.lib()
    assert lib.dsoft_siglip_g_bytes(None) == 0
    assert lib.dsoft_siglip_forward(*([None] * 9)) == -1
    assert lib.dsoft_siglip_backward(*([None] * 11)) == -1


UPSTREAM_INIT = ["self", "cache_labels", "rank", "world_size", "dist_impl"]
UPSTREAM_FORWARD = ["self", "image_features", "text_features", "logit_scale", "logit_bias", "output_dict"]


def test_signatures_match_upstream(pkg):
    init = inspect.signature(pkg.SigLipLoss.__init__).parameters
    assert list(init) == UPSTREAM_INIT + ["process_group"]
    assert [init[k].default for k in UPSTREAM_INIT[1:]] == [False, 0, 1, None]
    assert init["process_group"].default is None
    fwd = inspect.signature(pkg.SigLipLoss.forward).parameters
    assert list(fwd) == UPSTREAM_FORWARD
    assert fwd["logit_bias"].default is None and fwd["output_dict"].default is False
    if os.path.exists(REF_LOSS):
        ref = _ref_module()
        if hasattr(ref, "SigLipLoss"):
            assert list(inspect.signature(ref.SigLipLoss.__init__).parameters) == UPSTREAM_INIT
            assert list(inspect.signature(ref.SigLipLoss.forward).parameters)[:5] == UPSTREAM_FORWARD[:5]


def test_dist_impl_validation(pkg):
    assert pkg.SigLipLoss().dist_impl == "bidir"
    for impl in ("bidir", "shift", "reduce", "gather"):
        assert pkg.SigLipLoss(dist_impl=impl, rank=1, world_size=4).dist_impl == impl
    with pytest.raises(AssertionError):
        pkg.SigLipLoss(dist_impl="ring")


def test_forward_refuses_cpu_tensors(pkg):
    x = torch.randn(4, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        pkg.SigLipLoss()(x, x, torch.tensor(10.0), torch.tensor(-10.0))
    with pytest.raises(ValueError):
        pkg.SigLipLoss()(x, torch.randn(5, 8), torch.tensor(10.0))


def _fake_open_clip():
    class Clip:  # stand-ins for the fork's classes
        pass

    class Cyc:
        pass

    class Sig:
        pass

    loss = types.ModuleType("open_clip.loss")
    factory = types.ModuleType("open_clip.factory")
    train = types.ModuleType("open_clip_train.train")
    for m in (loss, factory):
        m.ClipLossWithDINOEnhancements, m.CyCLIPLoss, m.SigLipLoss = Clip, Cyc, Sig
    train.CyCLIPLoss, train.SigLipLoss = Cyc, Sig
    return types.SimpleNamespace(loss=loss, factory=factory), train, Sig


def test_install_and_uninstall(pkg, monkeypatch):
    oc, train, Sig = _fake_open_clip()
    monkeypatch.setitem(sys.modules, "open_clip_train.train", train)
    pkg.install_into_open_clip(oc)  # default: SigLIP stays upstream's
    assert oc.loss.SigLipLoss is Sig and oc.factory.SigLipLoss is Sig and train.SigLipLoss is Sig
    assert not hasattr(oc.loss, "_reference_SigLipLoss")
    assert oc.loss.ClipLossWithDINOEnhancements is pkg.ClipLossWithDINOEnhancements
    pkg.install_into_open_clip(oc, siglip=True)
    assert oc.loss.SigLipLoss is pkg.SigLipLoss and oc.factory.SigLipLoss is pkg.SigLipLoss
    assert train.SigLipLoss is pkg.SigLipLoss
    pkg.install_into_open_clip(oc, siglip=True)  # twice: the saved original is kept
    assert oc.loss._reference_SigLipLoss is Sig
    pkg.uninstall_from_open_clip(oc)
    assert oc.loss.SigLipLoss is Sig and oc.factory.SigLipLoss is Sig and train.SigLipLoss is Sig


# ---- the fp64 statement against the upstream recipes --------------------------------------------------------------
def _inputs(B, D, seed=0):
    g = torch.Generator().manual_seed(seed)
    img = torch.nn.functional.normalize(torch.randn(B, D, generator=g, dtype=torch.float64), dim=-1)
    txt = torch.nn.functional.normalize(img + 0.5 * torch.randn(B, D, generator=g, dtype=torch.float64), dim=-1)
    return img, txt


def test_statement_world1_is_the_plain_recipe():
    img, txt = _inputs(37, 16)
    logits = 10.0 * img @ txt.T - 10.0
    labels = 2 * torch.eye(37, dtype=torch.float64) - 1
    want = -torch.nn.functional.logsigmoid(labels * logits).sum() / 37
    assert float(siglip_ref.rank_loss(img, txt, 10.0, -10.0, 1, 0)) == pytest.approx(float(want), rel=1e-14)
    blk = siglip_ref.blocked(img, txt, 10.0, -10.0, rows=[slice(0, 37)], cols=[slice(5, 20)], block=8)
    full = siglip_ref.rank_grads(img, txt, 10.0, -10.0, 1)[0]
    assert blk["loss"] == pytest.approx(full["loss"], rel=1e-12)
    assert blk["d_scale"] == pytest.approx(full["d_scale"], rel=1e-12)
    assert blk["d_bias"] == pytest.approx(full["d_bias"], rel=1e-12)
    assert torch.allclose(blk["d_image"][0], full["d_image"], rtol=1e-12, atol=1e-15)
    assert torch.allclose(blk["d_text"][0], full["d_text"][5:20], rtol=1e-12, atol=1e-15)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _ref_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("dsoft_ref_loss_siglip", REF_LOSS)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _gather_recipe(img, txt, sc, bi, rank, world):
    """Upstream SigLipLoss.forward with dist_impl='gather', restated."""
    loss = siglip_ref.block_loss(img, txt, sc, bi)
    all_txt = torch.distributed.nn.all_gather(txt)
    for i in range(world):
        if i != rank:
            loss = loss + siglip_ref.block_loss(img, all_txt[i], sc, bi, negative_only=True)
    return loss


def _worker(rank, world, port, B, D, use_ref, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)

    img, txt = _inputs(B, D)
    b = B // world
    impls = ["gather"]
    ref = None
    if use_ref:
        ref = _ref_module()
        impls = ["bidir", "shift", "reduce", "gather"]
    out = {}
    for impl in impls:
        im = img[rank * b:(rank + 1) * b].clone().requires_grad_(True)
        tx = txt[rank * b:(rank + 1) * b].clone().requires_grad_(True)
        sc = torch.tensor(10.0, dtype=torch.float64, requires_grad=True)
        bi = torch.tensor(-10.0, dtype=torch.float64, requires_grad=True)
        if ref is None:
            loss = _gather_recipe(im, tx, sc, bi, rank, world)
        else:
            loss = ref.SigLipLoss(rank=rank, world_size=world, dist_impl=impl)(im, tx, sc, bi)
        loss.backward()
        out[impl] = dict(loss=float(loss.detach()), d_image=im.grad.clone(), d_text=tx.grad.clone(),
                         d_scale=float(sc.grad), d_bias=float(bi.grad))
    ret[rank] = out
    dist.barrier()
    dist.destroy_process_group()


def _check(outs, B, D, world):
    img, txt = _inputs(B, D)
    want = siglip_ref.rank_grads(img, txt, 10.0, -10.0, world)
    for r, per in enumerate(outs):
        for impl, o in per.items():
            w = want[r]
            assert o["loss"] == pytest.approx(w["loss"], rel=1e-12), (r, impl)
            assert o["d_scale"] == pytest.approx(w["d_scale"], rel=1e-10), (r, impl)
            assert o["d_bias"] == pytest.approx(w["d_bias"], rel=1e-10), (r, impl)
            for k in ("d_image", "d_text"):
                assert torch.allclose(o[k], w[k], rtol=1e-10, atol=1e-14), (r, impl, k)


def _spawn(world, B, D, use_ref):
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), B, D, use_ref, ret), nprocs=world, join=True)
    return [ret[r] for r in range(world)]


@pytest.mark.parametrize("world", [2, 3])
def test_statement_matches_gather_recipe_gloo(world):
    """Per-rank losses and gradients of the upstream `gather` recipe under gloo (all_gather with gradient)."""
    B, D = 12 * world, 16
    _check(_spawn(world, B, D, False), B, D, world)


@pytest.mark.skipif(not os.path.exists(REF_LOSS), reason="oracle/_ref/loss.py is not staged")
def test_statement_matches_staged_reference_every_dist_impl():
    if not hasattr(_ref_module(), "SigLipLoss"):
        pytest.skip("the staged reference has no SigLipLoss")
    B, D, world = 24, 16, 2
    _check(_spawn(world, B, D, True), B, D, world)
