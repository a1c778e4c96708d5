"""Weighted CE branch at world size > 1 (DSOFT_F_WEIGHTED, `weighted_scope="global"`), every rank on ONE GPU.

Rank r owns rows [r b, (r+1) b) of the global B x B problem; beta is the median of the row stds of all B rows.  As in
`test_gpu_multirank.py`, every rank is played through the C ABI on one device: `dsoft_pack` writes each rank's rows
into one shared `gathered` buffer, forward phase 5 runs per rank, the row-std blocks are all-gathered by hand (copied
into every rank's state), phase 6 runs per rank into its slice of the widened `lse_all`, and the backward runs per
rank.  Each rank is compared with fp64: the classic / soft terms from `oracle.rank_loss`, the weighted term from
`weighted_rows_ref.weighted_ce_global_rows` on the concatenated batch; loss terms 1e-4, gradients 1e-3 (max-abs and
L2 relative), d logit_scale 1e-3, beta 1e-5; the diagnostics against the row-block restatement
`weighted_rows_ref.weighted_ce_rows_branch`.
"""
import types

import pytest
import torch

from gpu_util import rel_err, synth
from test_gpu_multirank import seeded
from weighted_rows_ref import weighted_ce_global_rows, weighted_ce_rows_branch

pytestmark = pytest.mark.gpu

LOSS_RTOL, GRAD_RTOL, BETA_RTOL = 1e-4, 1e-3, 1e-5
LAM_W = 0.5
TEACHER_TEMP, TEXT_TEMP = 0.15, 0.02
RHO, C_CLIP = 0.2, 0.5
DBG_TOL = {"pos_frac_img": 2e-3, "neg_frac_img": 2e-3, "pos_frac_txt": 2e-3, "neg_frac_txt": 2e-3,
           "corr_rhat_dprob_img": 2e-3, "corr_rhat_dprob_txt": 2e-3}


def lambdas(soft):
    return (1.0, 0.5 if soft else 0.0, 0.5 if soft else 0.0, LAM_W)


def student_of(img, Dd, seed):
    """A raw (un-normalised) head output, bf16-representable like the module's straight-through rounding."""
    g = torch.Generator().manual_seed(seed)
    D = img.shape[1]
    mix = torch.randn(D, Dd, generator=g) / D ** 0.5
    return ((img @ mix) * 2.5 + 0.1 * torch.randn(img.shape[0], Dd, generator=g)).to(torch.bfloat16).float()


def oracle_ranks(oracle, img, txt, dino, student, scale, W, gwg, wsym, soft, gout=None):
    """Per-rank loss terms and gradients in fp64 (per-rank gradient convention of test_gpu_multirank.py), of
    sum_k gout[k] * term_k (default: of total_loss)."""
    lam = lambdas(soft)
    cfg = oracle.OracleConfig(lambda_original=lam[0], lambda_soft=lam[1], soft_mode="kl_teacher" if soft else "none",
                              teacher_temp=TEACHER_TEMP, soft_dino_to_text=soft, text_lambda=lam[2],
                              text_student_temp=TEXT_TEMP, world_size=W, local_loss=True, gather_with_grad=gwg,
                              rho=RHO, c_clip=C_CLIP, weight_text_symmetry=wsym)
    B = img.shape[0]
    b = B // W
    dt = torch.float64

    def leafs():
        im = img.to(dt).clone().requires_grad_(True)
        tx = txt.to(dt).clone().requires_grad_(True)
        sc = torch.tensor(float(scale), dtype=dt, requires_grad=True)
        st = None if student is None else student.to(dt).clone().requires_grad_(True)
        return im, tx, sc, st

    def rank_terms(im, tx, sc, st, r):
        t = oracle.rank_loss(im, tx, sc, dino.to(dt), st, cfg, rank=r)  # classic + soft (weighted raises at W > 1)
        rows = slice(r * b, (r + 1) * b)
        if gwg:
            li, lt = sc * (im @ tx.T), sc * (tx @ im.T)
        else:  # gathered copies detached: only this rank's rows carry gradient
            own = lambda x: torch.cat([x[:r * b].detach(), x[rows], x[(r + 1) * b:].detach()])
            li, lt = sc * (own(im) @ tx.detach().T), sc * (own(tx) @ im.detach().T)
        w = weighted_ce_global_rows(li, lt, dino.to(dt), rows, RHO, C_CLIP, wsym)
        t["weighted_loss"] = w["loss"]
        t["beta_img"], t["beta_txt"] = w["beta_img"], w["beta_txt"]
        t["total_loss"] = t["total_loss"] + LAM_W * w["loss"]
        return t

    out = []
    if gwg:
        im, tx, sc, st = leafs()
        per = [rank_terms(im, tx, sc, st, r) for r in range(W)]
        g_sc = [torch.autograd.grad(seeded(p, gout), sc, retain_graph=True)[0] for p in per]
        sum(seeded(p, gout) for p in per).backward()
        for r in range(W):
            rows = slice(r * b, (r + 1) * b)
            out.append(dict(terms=per[r], d_image=im.grad[rows], d_text=tx.grad[rows],
                            d_student=None if st is None else st.grad[rows], d_scale=float(g_sc[r])))
    else:
        for r in range(W):
            im, tx, sc, st = leafs()
            p = rank_terms(im, tx, sc, st, r)
            seeded(p, gout).backward()
            rows = slice(r * b, (r + 1) * b)
            out.append(dict(terms=p, d_image=im.grad[rows], d_text=tx.grad[rows],
                            d_student=None if st is None else st.grad[rows], d_scale=float(sc.grad)))
    return out


def cuda_ranks(img, txt, dino, student, scale, W, gwg, wsym, soft, want_dbg=True, gout=None):
    """Every rank of a W-rank job through the C ABI on cuda:0, the two collectives done by hand; gout: the six
    upstream gradients (default: d total_loss = 1)."""
    from dinosoft_b200 import _cabi
    from dinosoft_b200.loss import CudaBackend

    dev = torch.device("cuda", 0)
    be = CudaBackend()
    B, D = img.shape
    b = B // W
    flags = _cabi.DSOFT_F_WEIGHTED | _cabi.DSOFT_F_GMAT
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
    nr = plans[0].lse_rows
    assert nr == (5 if W == 1 else 5 + 3 * (2 if wsym else 1))
    lse_all = torch.empty((W, nr, b), dtype=torch.float32, device=dev)
    states = [torch.empty(pl.state_numel, dtype=torch.float32, device=dev) for pl in plans]
    scratch = [torch.empty(pl.fwd_scratch_numel, dtype=torch.float32, device=dev) for pl in plans]
    losses = [torch.empty(6, dtype=torch.float32, device=dev) for _ in plans]
    dbgs = [torch.empty(_cabi.DBG_N, dtype=torch.float32, device=dev) for _ in plans]
    for r, pl in enumerate(plans):
        be.forward(pl, gathered, ls, lam, states[r], scratch[r], lse_all[r], losses[r], dbgs[r] if want_dbg else None,
                   phase=5 if W > 1 else 0)
    if W > 1:
        off, n, _nd = plans[0].wsig
        assert all(pl.wsig == plans[0].wsig for pl in plans)
        full = torch.cat([states[r][off + r * n:off + (r + 1) * n] for r in range(W)])  # the all-gather
        for r, pl in enumerate(plans):
            states[r][off:off + W * n] = full
            be.forward(pl, gathered, ls, lam, states[r], scratch[r], lse_all[r], losses[r],
                       dbgs[r] if want_dbg else None, phase=6)
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
        out.append(dict(classic=float(lo[0]), soft=float(lo[3]), total=float(lo[4]), weighted=float(lo[5]),
                        dbg=dbgs[r].cpu(), d_image=d_image.cpu(), d_text=d_text.cpu(),
                        d_student=None if d_student is None else d_student.cpu(), d_scale=float(d_scale)))
    return out


def _inputs(W, b, soft, proj, D=128, Dd=192):
    B = W * b
    img, txt, dino = synth(41 + W, B, D, Dd)
    student = student_of(img, Dd, W) if (soft and proj) else None
    return img, txt, dino, student


@pytest.mark.parametrize("soft", [True, False], ids=["soft_text_proj", "clip_only"])
@pytest.mark.parametrize("gwg", [True, False], ids=["gather_grad", "no_gather_grad"])
@pytest.mark.parametrize("wsym", [True, False], ids=["wsym", "no_wsym"])
@pytest.mark.parametrize("W,b", [(2, 256), (4, 136), (8, 128)])
def test_every_rank_against_oracle(pkg, oracle, W, b, wsym, gwg, soft):
    from dinosoft_b200.loss import DBG_KEYS

    scale = 30.0
    img, txt, dino, student = _inputs(W, b, soft, True)
    want = oracle_ranks(oracle, img, txt, dino, student, scale, W, gwg, wsym, soft)
    got = cuda_ranks(img, txt, dino, student, scale, W, gwg, wsym, soft)
    idx = dict(DBG_KEYS)
    for r in range(W):
        o, ref = got[r], want[r]
        t = ref["terms"]
        for k, key in (("classic", "classic_loss"), ("soft", "soft_loss"), ("weighted", "weighted_loss"),
                       ("total", "total_loss")):
            assert o[k] == pytest.approx(float(t[key].detach()), rel=LOSS_RTOL, abs=1e-5), (r, k)
        assert float(o["dbg"][idx["beta_img"]]) == pytest.approx(t["beta_img"], rel=BETA_RTOL), (r, "beta_img")
        if wsym:
            assert float(o["dbg"][idx["beta_txt"]]) == pytest.approx(t["beta_txt"], rel=BETA_RTOL), (r, "beta_txt")
        worst = 0.0
        for k in ("d_image", "d_text", "d_student"):
            if ref[k] is None:
                continue
            linf, l2 = rel_err(o[k], ref[k])
            worst = max(worst, linf, l2)
            assert linf < GRAD_RTOL and l2 < GRAD_RTOL, (f"rank {r} of {W}", k, linf, l2)
        assert o["d_scale"] == pytest.approx(ref["d_scale"], rel=GRAD_RTOL, abs=1e-7), (r, "d_scale")
        print(f"[weighted multirank] W={W} b={b} wsym={wsym} gwg={gwg} soft={soft} rank {r}: worst grad {worst:.2e}")
    # diagnostics of every rank against the fp64 row-block restatement
    B = W * b
    for r in range(W):
        dbg = weighted_ce_rows_branch(img.double(), txt.double(), torch.tensor(scale, dtype=torch.float64),
                                      dino.double(), RHO, C_CLIP, wsym, slice(r * b, (r + 1) * b))[1]
        for k, i in DBG_KEYS:
            g, w = float(got[r]["dbg"][i]), float(dbg[k])
            assert g == pytest.approx(w, rel=DBG_TOL.get(k, 5e-4), abs=2e-5 if k.startswith("pc_err") else 1e-6), \
                (f"rank {r} of {W}, B={B}", k, g, w)


def test_fullsize_mean_over_ranks_matches_one_rank(pkg):
    """Global batch 32768 as 8 ranks of 4096 on one GPU against the world-size-1 CUDA result on the same batch:
    mean over ranks of weighted_loss to 1e-5, beta to 1e-6, every rank's d_image / d_text to W x the world-size-1
    gradient rows (1e-3)."""
    W, b, D, Dd = 8, 4096, 256, 384
    B = W * b
    img, txt, dino = synth(7, B, D, Dd)
    scale = 30.0
    one = cuda_ranks(img, txt, dino, None, scale, 1, True, True, True, want_dbg=True)[0]
    many = cuda_ranks(img, txt, dino, None, scale, W, True, True, True, want_dbg=True)
    from dinosoft_b200.loss import DBG_KEYS

    idx = dict(DBG_KEYS)
    mean_w = sum(o["weighted"] for o in many) / W
    assert mean_w == pytest.approx(one["weighted"], rel=1e-5)
    for r, o in enumerate(many):
        for k in ("beta_img", "beta_txt"):
            assert float(o["dbg"][idx[k]]) == pytest.approx(float(one["dbg"][idx[k]]), rel=1e-6), (r, k)
        rows = slice(r * b, (r + 1) * b)
        for k in ("d_image", "d_text"):
            linf, l2 = rel_err(o[k], W * one[k][rows])
            assert linf < GRAD_RTOL and l2 < GRAD_RTOL, (r, k, linf, l2)


def _module_run(pkg, img, txt, dino, scale, args, weighted_scope):
    dev = torch.device("cuda", 0)
    kw = {} if weighted_scope is None else {"weighted_scope": weighted_scope}
    loss = pkg.ClipLossWithDINOEnhancements(**kw)
    im = img.to(dev).requires_grad_(True)
    tx = txt.to(dev).requires_grad_(True)
    sc = torch.tensor(scale, device=dev, requires_grad=True)
    out = loss(im, tx, sc, dino.to(dev), args, output_dict=True)
    out["total_loss"].backward()
    return out, im.grad, tx.grad, sc.grad


@pytest.mark.parametrize("wsym", [True, False])
def test_world1_unchanged_by_keyword(pkg, wsym):
    """At world size 1 `weighted_scope="global"` runs exactly the same kernels: bitwise-equal outputs."""
    img, txt, dino = synth(5, 384, 128, 192)
    args = types.SimpleNamespace(use_projection=False, lambda_weighted=0.6, rho=RHO, c_clip=C_CLIP,
                                 weight_text_symmetry=wsym, lambda_soft=0.5, soft_mode="kl_teacher",
                                 soft_dino_to_text=True, text_lambda=0.5, text_student_temp=0.02)
    a = _module_run(pkg, img, txt, dino, 30.0, args, None)
    b = _module_run(pkg, img, txt, dino, 30.0, args, "global")
    for k in ("total_loss", "classic_loss", "soft_loss", "weighted_loss"):
        assert torch.equal(a[0][k], b[0][k]), k
    for k in a[0]["dbg"]:
        assert torch.equal(torch.as_tensor(a[0]["dbg"][k]), torch.as_tensor(b[0]["dbg"][k])), k
    for x, y in zip(a[1:], b[1:]):
        assert torch.equal(x, y)
