"""`ClipLossWithDINOEnhancements(..., weighted_scope="global")` over NCCL, one process per GPU, against the fp64
oracle of the concatenated batch (per-rank loss terms, beta, gradients) and the dbg dict (0-dim device tensors).
World size 2, and 8 where 8 GPUs are present; skipped with fewer than 2 GPUs."""
import os
import socket
import sys
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT
from gpu_util import rel_err, synth

pytestmark = pytest.mark.gpu

TEACHER_TEMP, TEXT_TEMP, RHO, C_CLIP, LAM_W = 0.15, 0.02, 0.2, 0.5, 0.5


def _args(wsym):
    return types.SimpleNamespace(use_projection=False, lambda_original=1.0, lambda_soft=0.5, soft_mode="kl_teacher",
                                 teacher_temp=TEACHER_TEMP, soft_dino_to_text=True, text_lambda=0.5,
                                 text_student_temp=TEXT_TEMP, lambda_weighted=LAM_W, rho=RHO, c_clip=C_CLIP,
                                 weight_text_symmetry=wsym)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, B, D, Dd, scale, wsym, gwg, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import dinosoft_b200 as pkg

    img, txt, dino = synth(23, B, D, Dd)
    b = B // world
    rows = slice(rank * b, (rank + 1) * b)
    dev = torch.device("cuda", rank)
    m = pkg.ClipLossWithDINOEnhancements(local_loss=True, gather_with_grad=gwg, rank=rank, world_size=world,
                                         weighted_scope="global")
    im = img[rows].to(dev).requires_grad_(True)
    tx = txt[rows].to(dev).requires_grad_(True)
    sc = torch.tensor(scale, device=dev, requires_grad=True)
    out = m(im, tx, sc, dino[rows].to(dev), _args(wsym), output_dict=True)
    dbg_ok = all((not torch.is_tensor(v)) or (v.dim() == 0 and v.device == dev) for v in out["dbg"].values())
    out["total_loss"].backward()
    torch.cuda.synchronize()
    ret[rank] = dict(total=float(out["total_loss"].detach()), classic=float(out["classic_loss"].detach()),
                     soft=float(out["soft_loss"].detach()), weighted=float(out["weighted_loss"].detach()),
                     beta_img=float(out["dbg"]["beta_img"]), beta_txt=float(out["dbg"]["beta_txt"]), dbg_ok=dbg_ok,
                     d_image=im.grad.cpu(), d_text=tx.grad.cpu(), d_scale=float(sc.grad))
    dist.barrier()
    dist.destroy_process_group()


def _check(oracle, world, b, wsym, gwg):
    from test_gpu_weighted_multirank import oracle_ranks

    B, D, Dd, scale = world * b, 128, 192, 30.0
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), B, D, Dd, scale, wsym, gwg, ret), nprocs=world, join=True)
    img, txt, dino = synth(23, B, D, Dd)
    want = oracle_ranks(oracle, img, txt, dino, None, scale, world, gwg, wsym, True)
    for r in range(world):
        o, ref = ret[r], want[r]
        t = ref["terms"]
        assert o["dbg_ok"], r
        for k, key in (("classic", "classic_loss"), ("soft", "soft_loss"), ("weighted", "weighted_loss"),
                       ("total", "total_loss")):
            assert o[k] == pytest.approx(float(t[key].detach()), rel=1e-4, abs=1e-5), (r, k)
        assert o["beta_img"] == pytest.approx(t["beta_img"], rel=1e-5)
        if wsym:
            assert o["beta_txt"] == pytest.approx(t["beta_txt"], rel=1e-5)
        for k in ("d_image", "d_text"):
            linf, l2 = rel_err(o[k], ref[k])
            print(f"[weighted-w{world}] rank {r} {k}: linf={linf:.2e} l2={l2:.2e}")
            assert linf < 1e-3 and l2 < 1e-3, (r, k, linf, l2)
        assert o["d_scale"] == pytest.approx(ref["d_scale"], rel=1e-3, abs=1e-7)


@pytest.mark.parametrize("wsym,gwg", [(True, True), (False, False)])
def test_two_gpu_weighted_global(oracle, wsym, gwg):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _check(oracle, 2, 512, wsym, gwg)


def test_eight_gpu_weighted_global(oracle):
    if torch.cuda.device_count() < 8:
        pytest.skip("needs 8 GPUs")
    _check(oracle, 8, 256, True, True)
