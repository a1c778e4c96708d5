"""World-size > 1 code path of the CUDA kernels on ONE GPU, through the C ABI (include/dsoft.h).

`tests/test_gpu_dist.py` needs two GPUs and is skipped on a one-GPU box.  The kernels themselves never talk to
another rank: a rank's launch reads the `gathered` table (all ranks' packed rows) and the all-gathered row
log-sum-exps.  This test plays every rank of a W-rank job on one device: `dsoft_pack` writes each rank's row
block into one `gathered` buffer (what the NCCL all-gather produces, loss.py:23-81), `dsoft_forward` runs per
rank into its slice of `lse_all`, and `dsoft_backward` runs per rank with the assembled `lse_all` - exactly the
sequence `_DinoSoftFn` drives, minus the two collectives.  Every rank (rank W-1 of 8 included) is compared with
the fp64 oracle: loss terms 1e-4, gradients 1e-3.

Matrix: W in {2, 4, 8} x soft scope {global, local} x gather_with_grad {on, off} x both backward paths.
"""
import ctypes as C

import pytest
import torch

from gpu_util import rel_err, synth

pytestmark = pytest.mark.gpu

LOSS_RTOL, GRAD_RTOL = 1e-4, 1e-3
LAMBDAS = (1.0, 0.5, 0.5, 0.0)  # lambda_original, lambda_soft, text_lambda, lambda_weighted
TEACHER_TEMP, TEXT_TEMP = 0.15, 0.02


TERMS = ("classic_loss", "soft_img", "soft_txt", "soft_loss", "total_loss", "weighted_loss")  # order of gout / losses


def seeded(terms, gout):
    """sum_k gout[k] * term_k: what the backward of upstream gradients gout differentiates (None: total_loss)."""
    if gout is None:
        return terms["total_loss"]
    return sum(float(g) * terms[k] for g, k in zip(gout, TERMS) if g != 0.0)


def oracle_ranks(oracle, img, txt, dino, student, scale, W, scope, gwg, gout=None):
    """Per-rank losses and gradients of the reference semantics (fp64), student given as a raw leaf tensor; the
    gradients are those of sum_k gout[k] * term_k (default: of total_loss)."""
    cfg = oracle.OracleConfig(lambda_original=LAMBDAS[0], lambda_soft=LAMBDAS[1], soft_mode="kl_teacher",
                              teacher_temp=TEACHER_TEMP, soft_dino_to_text=True, text_lambda=LAMBDAS[2],
                              text_student_temp=TEXT_TEMP, world_size=W, local_loss=True, gather_with_grad=gwg,
                              soft_scope=scope)
    B = img.shape[0]
    b = B // W
    dt = torch.float64
    out = []

    def leafs():
        im = img.to(dt).clone().requires_grad_(True)
        tx = txt.to(dt).clone().requires_grad_(True)
        sc = torch.tensor(float(scale), dtype=dt, requires_grad=True)
        st = None if student is None else student.to(dt).clone().requires_grad_(True)
        return im, tx, sc, st

    if gwg:
        # features: derivative of the SUM of all ranks' losses (all-gather backward = reduce-scatter);
        # logit_scale: each rank's own loss
        im, tx, sc, st = leafs()
        per = [oracle.rank_loss(im, tx, sc, dino.to(dt), st, cfg, rank=r) for r in range(W)]
        g_sc = [torch.autograd.grad(seeded(p, gout), sc, retain_graph=True)[0] for p in per]
        sum(seeded(p, gout) for p in per).backward()
        for r in range(W):
            rows = slice(r * b, (r + 1) * b)
            out.append(dict(terms=per[r], d_image=im.grad[rows], d_text=tx.grad[rows],
                            d_student=None if st is None else st.grad[rows], d_scale=float(g_sc[r])))
    else:
        for r in range(W):
            im, tx, sc, st = leafs()
            p = oracle.rank_loss(im, tx, sc, dino.to(dt), st, cfg, rank=r)
            seeded(p, gout).backward()
            rows = slice(r * b, (r + 1) * b)
            out.append(dict(terms=p, d_image=im.grad[rows], d_text=tx.grad[rows],
                            d_student=None if st is None else st.grad[rows], d_scale=float(sc.grad)))
    return out


def cuda_ranks(pkg, img, txt, dino, student, scale, W, scope, gwg, gmat, gout=None):
    """Every rank through the C ABI on cuda:0; gout: the six upstream gradients (default: d total_loss = 1)."""
    from dinosoft_b200 import _cabi
    from dinosoft_b200.loss import CudaBackend

    dev = torch.device("cuda", 0)
    be = CudaBackend()
    B, D = img.shape
    b = B // W
    flags = _cabi.DSOFT_F_SOFT | _cabi.DSOFT_F_TEXT
    if scope == "local":
        flags |= _cabi.DSOFT_F_SOFT_LOCAL
    if not gwg:
        flags |= _cabi.DSOFT_F_ROW_ONLY
    if gmat:
        flags |= _cabi.DSOFT_F_GMAT
    Dp = 0 if student is None else student.shape[1]
    plans = [be.plan(_cabi.Shape(b=b, world=W, rank=r, D=D, Dp=Dp, Dd=dino.shape[1], flags=flags,
                                 teacher_temp=TEACHER_TEMP, text_temp=TEXT_TEMP), dev) for r in range(W)]
    gathered = torch.empty((B, plans[0].row_elems), dtype=torch.bfloat16, device=dev)
    cu = lambda t: None if t is None else t.to(dev)
    for r, pl in enumerate(plans):  # every rank packs its own rows; the all-gather is the shared buffer itself
        rows = slice(r * b, (r + 1) * b)
        be.pack(pl, cu(img[rows]), cu(txt[rows]), cu(None if student is None else student[rows]), cu(dino[rows]),
                gathered)
    ls = torch.tensor([scale], dtype=torch.float32, device=dev)
    lse_all = torch.empty((W, 5, b), dtype=torch.float32, device=dev)
    states, losses = [], []
    for r, pl in enumerate(plans):
        st = torch.empty(pl.state_numel, dtype=torch.float32, device=dev)
        sc = torch.empty(pl.fwd_scratch_numel, dtype=torch.float32, device=dev)
        lo = torch.empty(6, dtype=torch.float32, device=dev)
        be.forward(pl, gathered, ls, LAMBDAS, st, sc, lse_all[r], lo)
        states.append(st)
        losses.append(lo)
    gout = torch.tensor([0.0, 0.0, 0.0, 0.0, 1.0, 0.0] if gout is None else list(gout), dtype=torch.float32,
                        device=dev)
    out = []
    for r, pl in enumerate(plans):
        scratch = torch.empty(pl.scratch_numel, dtype=torch.float32, device=dev)
        d_image = torch.empty((b, D), dtype=torch.float32, device=dev)
        d_text = torch.empty((b, D), dtype=torch.float32, device=dev)
        d_student = torch.empty((b, Dp), dtype=torch.float32, device=dev) if Dp else None
        d_scale = torch.empty(1, dtype=torch.float32, device=dev)
        be.backward(pl, gathered, states[r], scratch, lse_all, gout, LAMBDAS, d_image, d_text, d_student, d_scale)
        torch.cuda.synchronize()
        lo = losses[r].cpu()
        out.append(dict(classic=float(lo[0]), soft=float(lo[3]), total=float(lo[4]), d_image=d_image.cpu(),
                        d_text=d_text.cpu(), d_student=None if d_student is None else d_student.cpu(),
                        d_scale=float(d_scale)))
    return out


@pytest.mark.parametrize("gmat", [True, False], ids=["two_phase", "fused"])
@pytest.mark.parametrize("gwg", [True, False], ids=["gather_grad", "no_gather_grad"])
@pytest.mark.parametrize("scope", ["global", "local"])
@pytest.mark.parametrize("W,b,proj", [(2, 384, True), (4, 256, False), (8, 128, True), (8, 136, False)])
def test_every_rank_against_oracle(pkg, oracle, W, b, proj, scope, gwg, gmat):
    _run_case(pkg, oracle, W, b, proj, scope, gwg, gmat, 128, 192)


@pytest.mark.parametrize("gmat", [True, False], ids=["two_phase", "fused"])
def test_config4_dims_every_rank(pkg, oracle, gmat):
    """BASELINE config 4 feature dims (ViT-L/14: D = 768, DINOv2-L: 1024, no head, text-symmetric) at world 4:
    the CLIP kernels stream their row operand (K > 512), the gradient GEMMs run three 256-feature tiles."""
    _run_case(pkg, oracle, 4, 256, False, "global", True, gmat, 768, 1024)


def _run_case(pkg, oracle, W, b, proj, scope, gwg, gmat, D, Dd):
    B, scale = W * b, 30.0
    img, txt, dino = synth(31 + W, B, D, Dd)
    student = None
    if proj:  # a raw (un-normalised) head output, bf16-representable like the module's straight-through rounding
        g = torch.Generator().manual_seed(W)
        mix = torch.randn(D, Dd, generator=g) / D ** 0.5
        student = ((img @ mix) * 2.5 + 0.1 * torch.randn(B, Dd, generator=g)).to(torch.bfloat16).float()
    want = oracle_ranks(oracle, img, txt, dino, student, scale, W, scope, gwg)
    got = cuda_ranks(pkg, img, txt, dino, student, scale, W, scope, gwg, gmat)
    for r in range(W):
        o, ref = got[r], want[r]
        t = ref["terms"]
        for k, key in (("classic", "classic_loss"), ("soft", "soft_loss"), ("total", "total_loss")):
            assert o[k] == pytest.approx(float(t[key]), rel=LOSS_RTOL, abs=1e-5), (r, k)
        worst = 0.0
        for k in ("d_image", "d_text", "d_student"):
            if ref[k] is None:
                continue
            linf, l2 = rel_err(o[k], ref[k])
            worst = max(worst, linf, l2)
            assert linf < GRAD_RTOL and l2 < GRAD_RTOL, (f"rank {r} of {W}", k, linf, l2)
        assert o["d_scale"] == pytest.approx(ref["d_scale"], rel=GRAD_RTOL, abs=1e-7), (r, "d_scale")
        print(f"[multirank] W={W} b={b} scope={scope} gwg={gwg} gmat={gmat} rank {r}: worst grad err {worst:.2e}")
