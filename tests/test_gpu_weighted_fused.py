"""Weighted CE branch (DSOFT_F_WEIGHTED) on the fused backward: `dsoft_bwd_kernel<MODE_WCE_X>`, no DSOFT_F_GMAT.

- every rank of W = 2, 4 and 8 on one GPU through the C ABI against the fp64 statement of `weighted_rows_ref`
  (the oracle side of `test_gpu_weighted_multirank.py`), gradients and d logit_scale to 1e-3;
- fused against two-phase on the same inputs (W = 1 and every rank of W = 4), 5e-4;
- the module's OutOfMemoryError fallback for a weighted plan;
- global batch 65536 on one GPU with the allocator capped below the two-phase scratch;
- NCCL at W = 2 with `loss.GMAT = "never"` (skipped with fewer than 2 GPUs).
"""
import types

import pytest
import torch
import torch.multiprocessing as mp

from gpu_util import rel_err, synth
from test_gpu_weighted_multirank import (C_CLIP, GRAD_RTOL, LAM_W, LOSS_RTOL, RHO, TEACHER_TEMP, TEXT_TEMP, lambdas,
                                         oracle_ranks, student_of)

pytestmark = pytest.mark.gpu

PAIR_RTOL = 5e-4


def cuda_ranks(img, txt, dino, student, scale, W, gwg, wsym, soft, gmat, gout=None):
    """Every rank of a W-rank weighted job through the C ABI on cuda:0 (the two collectives done by hand), with or
    without DSOFT_F_GMAT, for the six upstream gradients gout (default: d total_loss = 1).  Returns per rank the
    losses and the four gradients."""
    from dinosoft_b200 import _cabi
    from dinosoft_b200.loss import CudaBackend

    dev = torch.device("cuda", 0)
    be = CudaBackend()
    B, D = img.shape
    b = B // W
    flags = _cabi.DSOFT_F_WEIGHTED | (_cabi.DSOFT_F_GMAT if gmat else 0)
    if wsym:
        flags |= _cabi.DSOFT_F_WSYM
    if soft:
        flags |= _cabi.DSOFT_F_SOFT | _cabi.DSOFT_F_TEXT
    if not gwg and W > 1:
        flags |= _cabi.DSOFT_F_ROW_ONLY
    Dp = student.shape[1] if (soft and student is not None) else 0
    lam = lambdas(soft)
    plans = [be.plan(_cabi.Shape(b=b, world=W, rank=r, D=D, Dp=Dp, Dd=dino.shape[1], flags=flags,
                                 teacher_temp=TEACHER_TEMP if soft else 0.0, text_temp=TEXT_TEMP if soft else 0.0,
                                 rho=RHO, c_clip=C_CLIP), dev) for r in range(W)]
    gathered = torch.empty((B, plans[0].row_elems), dtype=torch.bfloat16, device=dev)
    cu = lambda t: None if t is None else t.to(dev)
    for r, pl in enumerate(plans):
        rows = slice(r * b, (r + 1) * b)
        be.pack(pl, cu(img[rows]), cu(txt[rows]), cu(student[rows]) if Dp else None, cu(dino[rows]), gathered)
    ls = torch.tensor([scale], dtype=torch.float32, device=dev)
    lse_all = torch.empty((W, plans[0].lse_rows, b), dtype=torch.float32, device=dev)
    states = [torch.empty(pl.state_numel, dtype=torch.float32, device=dev) for pl in plans]
    scratch = [torch.empty(pl.fwd_scratch_numel, dtype=torch.float32, device=dev) for pl in plans]
    losses = [torch.empty(6, dtype=torch.float32, device=dev) for _ in plans]
    for r, pl in enumerate(plans):
        be.forward(pl, gathered, ls, lam, states[r], scratch[r], lse_all[r], losses[r], None, phase=5 if W > 1 else 0)
    if W > 1:
        off, n, _nd = plans[0].wsig
        full = torch.cat([states[r][off + r * n:off + (r + 1) * n] for r in range(W)])  # the all-gather
        for r, pl in enumerate(plans):
            states[r][off:off + W * n] = full
            be.forward(pl, gathered, ls, lam, states[r], scratch[r], lse_all[r], losses[r], None, phase=6)
    gout = torch.tensor([0.0, 0.0, 0.0, 0.0, 1.0, 0.0] if gout is None else list(gout), dtype=torch.float32,
                        device=dev)
    out = []
    for r, pl in enumerate(plans):
        sc = torch.empty(pl.scratch_numel, dtype=torch.float32, device=dev)
        d_image = torch.empty((b, D), dtype=torch.float32, device=dev)
        d_text = torch.empty((b, D), dtype=torch.float32, device=dev)
        d_student = torch.empty((b, Dp), dtype=torch.float32, device=dev) if Dp else None
        d_scale = torch.empty(1, dtype=torch.float32, device=dev)
        be.backward(pl, gathered, states[r], sc, lse_all, gout, lam, d_image, d_text, d_student, d_scale)
        torch.cuda.synchronize()
        lo = losses[r].cpu()
        out.append(dict(total=float(lo[4]), weighted=float(lo[5]), d_image=d_image.cpu(), d_text=d_text.cpu(),
                        d_student=None if d_student is None else d_student.cpu(), d_scale=float(d_scale)))
    return out


@pytest.mark.parametrize("soft", [True, False], ids=["soft_text_proj", "clip_only"])
@pytest.mark.parametrize("gwg", [True, False], ids=["gather_grad", "no_gather_grad"])
@pytest.mark.parametrize("wsym", [True, False], ids=["wsym", "no_wsym"])
@pytest.mark.parametrize("W,b", [(2, 256), (4, 136), (8, 128)])
def test_fused_every_rank_against_oracle(oracle, W, b, wsym, gwg, soft):
    scale = 30.0
    img, txt, dino = synth(41 + W, W * b, 128, 192)
    student = student_of(img, 192, W) if soft else None
    want = oracle_ranks(oracle, img, txt, dino, student, scale, W, gwg, wsym, soft)
    got = cuda_ranks(img, txt, dino, student, scale, W, gwg, wsym, soft, gmat=False)
    for r in range(W):
        o, ref = got[r], want[r]
        t = ref["terms"]
        assert o["weighted"] == pytest.approx(float(t["weighted_loss"].detach()), rel=LOSS_RTOL, abs=1e-5), r
        assert o["total"] == pytest.approx(float(t["total_loss"].detach()), rel=LOSS_RTOL, abs=1e-5), r
        worst = 0.0
        for k in ("d_image", "d_text", "d_student"):
            if ref[k] is None:
                continue
            linf, l2 = rel_err(o[k], ref[k])
            worst = max(worst, linf, l2)
            assert linf < GRAD_RTOL and l2 < GRAD_RTOL, (f"rank {r} of {W}", k, linf, l2)
        assert o["d_scale"] == pytest.approx(ref["d_scale"], rel=GRAD_RTOL, abs=1e-7), (r, "d_scale")
        print(f"[weighted fused] W={W} b={b} wsym={wsym} gwg={gwg} soft={soft} rank {r}: worst grad {worst:.2e}")


@pytest.mark.parametrize("wsym", [True, False], ids=["wsym", "no_wsym"])
@pytest.mark.parametrize("W,b,gwg", [(1, 1024, True), (4, 256, True), (4, 256, False)])
def test_fused_matches_two_phase(W, b, gwg, wsym):
    scale = 30.0
    img, txt, dino = synth(17 + W, W * b, 256, 384)
    student = student_of(img, 256, 3)
    two = cuda_ranks(img, txt, dino, student, scale, W, gwg, wsym, True, gmat=True)
    one = cuda_ranks(img, txt, dino, student, scale, W, gwg, wsym, True, gmat=False)
    for r in range(W):
        assert one[r]["total"] == two[r]["total"], r  # the forward does not depend on the backward form
        errs = {}
        for k in ("d_image", "d_text", "d_student"):
            errs[k] = max(rel_err(one[r][k], two[r][k]))
            assert errs[k] < PAIR_RTOL, (r, k, errs[k])
        errs["d_scale"] = abs(one[r]["d_scale"] - two[r]["d_scale"]) / abs(two[r]["d_scale"])
        assert errs["d_scale"] < PAIR_RTOL, (r, errs["d_scale"])
        print(f"[fused vs two-phase] W={W} gwg={gwg} wsym={wsym} rank {r}: " +
              " ".join(f"{k}={v:.2e}" for k, v in errs.items()))


def _module_args(**kw):
    base = dict(use_projection=True, projection_type="mlp", lambda_soft=0.5, soft_mode="kl_teacher",
                soft_dino_to_text=True, text_lambda=0.5, text_student_temp=0.02, teacher_temp=0.15,
                lambda_original=1.0, lambda_weighted=0.5, rho=RHO, c_clip=C_CLIP, weight_text_symmetry=True)
    base.update(kw)
    return types.SimpleNamespace(**base)


def test_oom_fallback_for_weighted_plan(pkg):
    """Two-phase backward chosen in the forward, its scratch cannot be allocated: a weighted plan now falls back to
    the fused backward on the same saved state (before this, the OutOfMemoryError was re-raised)."""
    from dinosoft_b200 import _cabi
    from dinosoft_b200 import loss as loss_mod

    img, txt, dino = (x.cuda() for x in synth(9, 384, 128, 192))
    args = _module_args()
    old = loss_mod.GMAT
    grads = []
    try:
        for sabotage in (False, True):
            loss_mod.GMAT = "auto"
            m = pkg.ClipLossWithDINOEnhancements()
            torch.manual_seed(0)
            m.init_proj(img.shape[1], dino.shape[1], img.device, "mlp")
            im = img.clone().requires_grad_(True)
            tx = txt.clone().requires_grad_(True)
            sc = torch.tensor(20.0, device="cuda", requires_grad=True)
            out = m(im, tx, sc, dino, args, output_dict=True)["total_loss"]
            plan = next(p for p in loss_mod._cuda_backend._plans.values()
                        if p.shape.b == 384 and p.shape.flags & _cabi.DSOFT_F_GMAT
                        and p.shape.flags & _cabi.DSOFT_F_WEIGHTED)
            keep = plan.scratch_numel
            if sabotage:
                plan.scratch_numel = 1 << 42  # 16 TiB of fp32: torch raises OutOfMemoryError
            try:
                out.backward()
            finally:
                plan.scratch_numel = keep
            torch.cuda.synchronize()
            grads.append((im.grad.clone(), tx.grad.clone(), sc.grad.clone(),
                          m.image_to_dino_proj[0].weight.grad.clone()))
    finally:
        loss_mod.GMAT = old
        loss_mod._gmat_decisions.clear()
    for k, (a, b) in enumerate(zip(grads[0], grads[1])):
        linf, l2 = rel_err(b, a)
        print(f"[weighted oom fallback] grad {k}: linf={linf:.2e} l2={l2:.2e}")
        assert linf < PAIR_RTOL and l2 < PAIR_RTOL, (k, linf, l2)


def test_global_batch_65536_under_memory_cap(pkg):
    """Global batch 65536 on one GPU, default soft + text + MLP head, lambda_weighted = 0.5 with weight_text_symmetry,
    `auto`, with this process's allocator capped so that the two-phase backward scratch (~30 GB with the forward
    part) cannot be allocated and the fused one (~5 GB) can: the step completes through the OutOfMemoryError
    fallback, and the feature gradients are linear in the upstream gradient."""
    from dinosoft_b200 import loss as loss_mod

    B, D, Dd = 65536, 512, 768
    dev = torch.device("cuda", 0)
    args = _module_args()
    img, txt, dino = synth(3, B, D, Dd, device=dev)
    torch.cuda.empty_cache()
    total = torch.cuda.get_device_properties(dev).total_memory
    old_gmat = loss_mod.GMAT
    loss_mod.GMAT = "auto"
    cap = (torch.cuda.memory_allocated(dev) + 20 * 2 ** 30) / total  # room for ~20 GB more than the inputs
    torch.cuda.set_per_process_memory_fraction(cap, dev)
    grads = []
    try:
        m = pkg.ClipLossWithDINOEnhancements()
        torch.manual_seed(0)
        m.init_proj(D, Dd, dev, "mlp")
        for mult in (1.0, 2.0):
            im = img.clone().requires_grad_(True)
            tx = txt.clone().requires_grad_(True)
            sc = torch.tensor(20.0, device=dev, requires_grad=True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = m(im, tx, sc, dino, args, output_dict=True)
            (mult * out["total_loss"]).backward()
            torch.cuda.synchronize()
            assert torch.isfinite(im.grad).all() and torch.isfinite(tx.grad).all() and torch.isfinite(sc.grad)
            grads.append((im.grad, tx.grad))
            del out, im, tx, sc
        print(f"[weighted B=65536 capped] fraction {cap:.3f} of {total / 2 ** 30:.0f} GiB, "
              f"peak {torch.cuda.max_memory_allocated(dev) / 2 ** 30:.1f} GiB")
    finally:
        torch.cuda.set_per_process_memory_fraction(1.0, dev)
        loss_mod.GMAT = old_gmat
        loss_mod._gmat_decisions.clear()
    for a, b in zip(*grads):
        linf, l2 = rel_err(b, 2.0 * a)
        assert linf < 1e-5 and l2 < 1e-5, (linf, l2)


def _nccl_worker(rank, world, port, B, D, Dd, scale, wsym, gwg, ret):
    from dinosoft_b200 import loss as loss_mod
    from test_gpu_weighted_dist import _worker

    loss_mod.GMAT = "never"
    _worker(rank, world, port, B, D, Dd, scale, wsym, gwg, ret)


@pytest.mark.parametrize("wsym,gwg", [(True, True), (False, False)])
def test_two_gpu_weighted_global_fused(oracle, wsym, gwg):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from test_gpu_weighted_dist import _free_port

    world, b, D, Dd, scale = 2, 512, 128, 192, 30.0
    B = world * b
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_nccl_worker, args=(world, _free_port(), B, D, Dd, scale, wsym, gwg, ret), nprocs=world, join=True)
    img, txt, dino = synth(23, B, D, Dd)
    want = oracle_ranks(oracle, img, txt, dino, None, scale, world, gwg, wsym, True)
    for r in range(world):
        o, ref = ret[r], want[r]
        assert o["weighted"] == pytest.approx(float(ref["terms"]["weighted_loss"].detach()), rel=1e-4, abs=1e-5)
        for k in ("d_image", "d_text"):
            linf, l2 = rel_err(o[k], ref[k])
            assert linf < 1e-3 and l2 < 1e-3, (r, k, linf, l2)
        assert o["d_scale"] == pytest.approx(ref["d_scale"], rel=1e-3, abs=1e-7)
