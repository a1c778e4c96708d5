"""Backward parity at the upstream gradients training really sends, against fp64.

Training does not seed the loss backward with 1: open_clip's `--precision amp` goes through `torch.amp.GradScaler`,
whose initial scale is 2^16 and which doubles it every 2000 clean steps; loss terms are also weighted one by one.  The
contract checked here: the gradients are the fp64 gradients of  sum_k gout[k] * term_k  for any gout, at every
magnitude training produces.  The backward carries the upstream gradient in two ways, both exercised:
- applied in fp32 after the fp16 logit-gradient matrices (CLIP, soft terms, SigLIP): exactly linear in the seed;
- inside the fp16 matrix times a power of two chosen on the device (DistillClipLoss, the weighted CE branch).

(a) module, world 1, both backward paths: seeds u in {2^-12, 1, 3, 2^16, 2^20} of total_loss on four configurations;
    every gradient finite, within the bar of u x the fp64 gradient, and for power-of-two u equal to u x grads(1);
(b) per-term seeds: through the module (classic, soft, weighted, total) and through the C ABI with all six entries of
    gout on every rank of W = 4 (soft_imgimg and soft_texttext are reachable only there);
(c) SigLipLoss, DistillClipLoss and CyCLIPLoss at GradScaler-sized and tiny seeds;
(d) one real GradScaler step under fp16 autocast on the weighted configuration: no step skipped;
(e) CUDA-graph replay: the captured backward follows the seed of each replay (GradScaler's back-off 2^16 -> 2^15).

Bars: the suite's, loss 1e-4 and gradients 1e-3 relative (max-abs over max-abs, and L2); d logit_scale 1e-3 relative;
linearity 1e-6 max-abs relative.  Each fp64 reference is computed once at seed 1 and scaled: it is linear.
"""
import math
import types

import pytest
import torch

import distill_ref
import siglip_ref
import test_gpu_multirank as multirank
import test_gpu_weighted_fused as wfused
import test_gpu_weighted_multirank as wmulti
from gpu_util import head_params_of, make_args, oracle_cfg, rel_err, synth

pytestmark = pytest.mark.gpu

LOSS_RTOL, GRAD_RTOL, LIN_RTOL = 1e-4, 1e-3, 1e-6
SEEDS = (2.0 ** -12, 1.0, 3.0, 2.0 ** 16, 2.0 ** 20)
DEV = "cuda"

_WEIGHTED = dict(lambda_weighted=0.6, rho=0.2, c_clip=0.5)
CONFIGS = {  # name: B, D, Dd, logit scale, input seed, loss args
    # the default workload: soft + text terms, MLP head
    "soft_text_mlp": (1024, 256, 384, 30.0, 1, make_args(use_projection=True)),
    # the inputs of test_weighted_ce_branch: everything on (classic + soft + weighted with weight_text_symmetry, head)
    "weighted_sym_soft_mlp": (256, 128, 192, 30.0, 11,
                              make_args(use_projection=True, weight_text_symmetry=True, **_WEIGHTED)),
    # weighted CE next to the classic CE only, several column splits, sharp rows (scale 60)
    "weighted_clip_only": (2048, 128, 192, 60.0, 11,
                           make_args(lambda_soft=0.0, soft_mode="none", **_WEIGHTED)),
    # flat rows (scale 14.29): many small logit-gradient entries, the first to leave fp16 at a small seed
    "weighted_flat_b4096": (4096, 512, 768, 14.2857, 11,
                            make_args(lambda_soft=0.0, soft_mode="none", weight_text_symmetry=True, **_WEIGHTED)),
}


@pytest.fixture(params=["two_phase", "fused"])
def backward_path(request, pkg):
    """Both backward implementations (test_gpu_parity.py's switch): the two-phase one (fp16 logit-gradient matrices +
    gradient GEMMs, DSOFT_F_GMAT) and the fused one."""
    from dinosoft_b200 import loss as loss_mod

    old = loss_mod.GMAT
    loss_mod.GMAT = "always" if request.param == "two_phase" else "never"
    yield request.param
    loss_mod.GMAT = old


def run_module(pkg, inputs, scale, args, seed_of, head_seed=7):
    """Forward through the module, backward of seed_of(output dict).  Returns the output dict, the gradients (fp64 on
    the host: d_image, d_text, d_logit_scale, d_student with a head, head_<param>), the student values the kernels used
    and the head parameters."""
    img, txt, dino = inputs
    loss = pkg.ClipLossWithDINOEnhancements()
    im = img.to(DEV).requires_grad_(True)
    tx = txt.to(DEV).requires_grad_(True)
    sc = torch.tensor(scale, device=DEV, requires_grad=True)
    grabbed, hook, head = {}, None, None
    if args.use_projection:
        torch.manual_seed(head_seed)
        loss.init_proj(img.shape[1], dino.shape[1], DEV, args.projection_type)
        hook = loss.image_to_dino_proj.register_forward_hook(
            lambda mod, inp, o: (grabbed.__setitem__("student", o.detach().to(torch.bfloat16).float().cpu()),
                                 o.register_hook(lambda g: grabbed.__setitem__("d_student", g.detach().clone())))
            and None)
    out = loss(im, tx, sc, dino.to(DEV), args, output_dict=True)
    seed_of(out).backward()
    torch.cuda.synchronize()
    grads = {"d_image": im.grad, "d_text": tx.grad, "d_logit_scale": sc.grad.reshape(())}
    if hook is not None:
        hook.remove()
        grads["d_student"] = grabbed["d_student"]
        params = head_params_of(loss.image_to_dino_proj, args.projection_type)
        head = {k: p.detach().cpu() for k, p in params.items()}
        grads.update({"head_" + k: p.grad for k, p in params.items()})
    grads = {k: v.detach().double().cpu() for k, v in grads.items()}
    return out, grads, grabbed.get("student"), head


_MODULE_REF = {}


def module_ref(oracle, name, student, head):
    """fp64 losses and gradients of total_loss (seed 1) for configuration `name`, computed once.  The oracle is handed
    the student VALUES the kernels used (their fp32 head output rounded to bf16), as check_against_oracle does."""
    if name not in _MODULE_REF:
        B, D, Dd, scale, seed, args = CONFIGS[name]
        img, txt, dino = synth(seed, B, D, Dd)
        cfg = oracle_cfg(oracle, args, round_student_bf16=True)
        r = oracle.loss_and_grads(img, txt, scale, dino, cfg, proj_params=head, projection_type=args.projection_type,
                                  dtype=torch.float64, student_values=student)["ranks"][0]
        ref = {"d_image": r["d_image"], "d_text": r["d_text"],
               "d_logit_scale": torch.tensor(r["d_logit_scale"], dtype=torch.float64)}
        if head is not None:
            ref["d_student"] = r["d_student"]
            ref.update({"head_" + k: v for k, v in r["d_proj"].items() if v is not None})
        losses = {k: r[k] for k in ("total_loss", "classic_loss", "soft_loss", "weighted_loss")}
        _MODULE_REF[name] = (losses, ref)
    return _MODULE_REF[name]


def grad_problems(tag, got, ref, u):
    """Bar of every gradient in `ref` against u x ref: a list of failure lines (empty: all within the bar)."""
    bad = []
    for k, want in ref.items():
        g = got[k]
        if not torch.isfinite(g).all():
            bad.append(f"{tag} {k}: {int((~torch.isfinite(g)).sum())} non-finite entries")
            continue
        w = u * want.double()
        if g.dim() == 0:
            err = abs(float(g) - float(w))
            ok = err <= GRAD_RTOL * abs(float(w)) + 1e-7 * u
            print(f"[upstream] {tag} {k}: got={float(g):.6e} ref={float(w):.6e}")
            if not ok:
                bad.append(f"{tag} {k}: got {float(g):.6e}, fp64 {float(w):.6e}")
            continue
        linf, l2 = rel_err(g, w)
        print(f"[upstream] {tag} {k}: linf={linf:.2e} l2={l2:.2e}")
        if not (linf < GRAD_RTOL and l2 < GRAD_RTOL):
            bad.append(f"{tag} {k}: linf={linf:.2e} l2={l2:.2e} against fp64")
    return bad


def linearity_problems(tag, runs):
    """For power-of-two seeds u: grads(u) == u * grads(1) to LIN_RTOL (max-abs relative); prints the worst ratio."""
    bad = []
    base = runs[1.0]
    for u, g in runs.items():
        if u == 1.0 or math.frexp(u)[0] != 0.5:
            continue
        worst, exact = 0.0, True
        for k, b in base.items():
            if not (torch.isfinite(g[k]).all() and torch.isfinite(b).all()):
                bad.append(f"{tag} u={u:g} {k}: non-finite, linearity not measurable")
                continue
            w = u * b
            err = (g[k] - w).abs().max().item() / max(w.abs().max().item(), 1e-300)
            exact = exact and torch.equal(g[k], w)
            worst = max(worst, err)
            if err >= LIN_RTOL:
                bad.append(f"{tag} u={u:g} {k}: |grads(u) - u grads(1)| / |u grads(1)| = {err:.2e}")
        print(f"[upstream] {tag} u={u:g}: worst linearity ratio {worst:.2e}{' (bitwise)' if exact else ''}")
    return bad


# --------------------------------------------------------------------------- (a) magnitude sweep through the module
@pytest.mark.parametrize("name", list(CONFIGS))
def test_seed_magnitude_sweep(pkg, oracle, backward_path, name):
    B, D, Dd, scale, seed, args = CONFIGS[name]
    inputs = synth(seed, B, D, Dd)
    runs, student, head = {}, None, None
    for u in SEEDS:
        out, runs[u], student, head = run_module(pkg, inputs, scale, args, lambda o, u=u: u * o["total_loss"])
    losses, ref = module_ref(oracle, name, student, head)
    for k, want in losses.items():  # the forward does not see the seed; checked once
        assert float(out[k].detach()) == pytest.approx(want, rel=LOSS_RTOL, abs=1e-5), k
    bad = []
    for u, g in runs.items():
        bad += grad_problems(f"{name} {backward_path} u={u:g}", g, ref, u)
    bad += linearity_problems(f"{name} {backward_path}", runs)
    assert not bad, "\n".join(bad)


# --------------------------------------------------------------------------- (b) per-term seeds
COMBO = {"classic_loss": 0.7, "soft_loss": -1.3, "weighted_loss": 2.1, "total_loss": 0.4}
GOUT6 = (0.7, -0.4, 1.1, -1.3, 0.4, 2.1)  # classic, soft_imgimg, soft_texttext, soft, total, weighted


@pytest.mark.parametrize("name", ["soft_text_mlp", "weighted_sym_soft_mlp"])
def test_per_term_seeds_module(pkg, oracle, backward_path, name):
    """(0.7 classic - 1.3 soft + 2.1 weighted + 0.4 total).backward() against fp64 autograd of the same combination of
    oracle.rank_loss's terms (no head: the student is the image feature)."""
    B, D, Dd, scale, seed, args = CONFIGS[name]
    args = types.SimpleNamespace(**{**vars(args), "use_projection": False})
    img, txt, dino = synth(seed, B, D, Dd)
    _, got, _, _ = run_module(pkg, (img, txt, dino), scale, args,
                              lambda o: sum(c * o[k] for k, c in COMBO.items()))
    dt = torch.float64
    im = img.to(dt).requires_grad_(True)
    tx = txt.to(dt).requires_grad_(True)
    sc = torch.tensor(scale, dtype=dt, requires_grad=True)
    terms = oracle.rank_loss(im, tx, sc, dino.to(dt), None, oracle_cfg(oracle, args))
    sum(c * terms[k] for k, c in COMBO.items()).backward()
    ref = {"d_image": im.grad, "d_text": tx.grad, "d_logit_scale": sc.grad}
    bad = grad_problems(f"{name} {backward_path} combo", got, ref, 1.0)
    assert not bad, "\n".join(bad)


def _rank_problems(tag, got, want, u, keys=("d_image", "d_text", "d_student")):
    bad = []
    for r, (o, ref) in enumerate(zip(got, want)):
        g = {k: o[k].double() for k in keys if ref.get(k) is not None}
        g["d_logit_scale"] = torch.tensor(o["d_scale"], dtype=torch.float64)
        w = {k: ref[k] for k in keys if ref.get(k) is not None}
        w["d_logit_scale"] = torch.tensor(ref["d_scale"], dtype=torch.float64)
        bad += grad_problems(f"{tag} rank {r}", g, w, u)
    return bad


@pytest.mark.parametrize("gmat", [True, False], ids=["two_phase", "fused"])
@pytest.mark.parametrize("gwg", [True, False], ids=["gather_grad", "no_gather_grad"])
def test_six_upstream_gradients_every_rank(pkg, oracle, gwg, gmat):
    """All six entries of gout through the C ABI, every rank of W = 4 (soft + text, global soft scope), at u = 1 and
    u = 2^16, against the fp64 gradients of sum_k gout[k] * term_k."""
    W, b, D, Dd, scale = 4, 256, 128, 192, 30.0
    img, txt, dino = synth(31 + W, W * b, D, Dd)
    want = multirank.oracle_ranks(oracle, img, txt, dino, None, scale, W, "global", gwg, gout=GOUT6)
    bad = []
    for u in (1.0, 2.0 ** 16):
        got = multirank.cuda_ranks(pkg, img, txt, dino, None, scale, W, "global", gwg, gmat,
                                   gout=[u * g for g in GOUT6])
        bad += _rank_problems(f"W={W} gwg={gwg} gmat={gmat} u={u:g}", got, want, u)
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("gmat", [True, False], ids=["two_phase", "fused"])
def test_six_upstream_gradients_weighted_every_rank(oracle, gmat):
    """The same for the weighted CE branch at W = 4 (weighted_scope="global", weight_text_symmetry, soft + text,
    student head output), at u = 1 and u = 2^16."""
    W, b, scale = 4, 136, 30.0
    img, txt, dino, student = wmulti._inputs(W, b, True, True)
    want = wmulti.oracle_ranks(oracle, img, txt, dino, student, scale, W, True, True, True, gout=GOUT6)
    bad = []
    for u in (1.0, 2.0 ** 16):
        got = wfused.cuda_ranks(img, txt, dino, student, scale, W, True, True, True, gmat,
                                gout=[u * g for g in GOUT6])
        bad += _rank_problems(f"weighted W={W} gmat={gmat} u={u:g}", got, want, u)
    assert not bad, "\n".join(bad)


# --------------------------------------------------------------------------- (c) the other losses
_SIGLIP_REF = {}


@pytest.mark.parametrize("u", [2.0 ** -12, 2.0 ** 16, 2.0 ** 20])
def test_siglip_seed_magnitude(pkg, u):
    B, D, s, beta = 1000, 768, 10.0, -10.0
    img, txt, _ = synth(B + D, B, D, 8)
    img, txt = img.to(DEV), txt.to(DEV)
    if "ref" not in _SIGLIP_REF:
        _SIGLIP_REF["ref"] = siglip_ref.rank_grads(img.double(), txt.double(), s, beta, 1)[0]
    ref = _SIGLIP_REF["ref"]
    im, tx = img.clone().requires_grad_(True), txt.clone().requires_grad_(True)
    sc = torch.tensor(s, device=DEV, requires_grad=True)
    bi = torch.tensor(beta, device=DEV, requires_grad=True)
    (u * pkg.SigLipLoss()(im, tx, sc, bi)).backward()
    torch.cuda.synchronize()
    got = {"d_image": im.grad.double().cpu(), "d_text": tx.grad.double().cpu(),
           "d_logit_scale": sc.grad.double().cpu(), "d_bias": bi.grad.double().cpu()}
    want = {"d_image": ref["d_image"].cpu(), "d_text": ref["d_text"].cpu(),
            "d_logit_scale": torch.tensor(ref["d_scale"], dtype=torch.float64),
            "d_bias": torch.tensor(ref["d_bias"], dtype=torch.float64)}
    bad = grad_problems(f"siglip u={u:g}", got, want, u)
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("u", [2.0 ** 16, 2.0 ** -12])
def test_distill_seed_magnitude(pkg, u):
    """(g_c, g_d) = u (0.3, 1.7): the device-chosen G scale of DistillClipLoss far from the (0.3, 1.7) case."""
    B, D, Dt, s, st = 2049, 512, 768, 14.29, 100.0
    img, txt, _ = synth(B + D, B, D, 8)
    dimg, dtxt, _ = synth(B + D + 1, B, Dt, 8)
    gc, gd = u * 0.3, u * 1.7
    ref = distill_ref.rank_grads(img.double(), txt.double(), dimg.double(), dtxt.double(), s, st, 1, gc=gc, gd=gd)[0]
    im, tx = img.to(DEV).requires_grad_(True), txt.to(DEV).requires_grad_(True)
    sc = torch.tensor(s, device=DEV, requires_grad=True)
    c, d = pkg.DistillClipLoss()(im, tx, sc, dimg.to(DEV), dtxt.to(DEV), torch.tensor(st, device=DEV))
    (gc * c + gd * d).backward()
    torch.cuda.synchronize()
    got = {"d_image": im.grad.double().cpu(), "d_text": tx.grad.double().cpu(), "d_logit_scale": sc.grad.double().cpu()}
    want = {"d_image": ref["d_image"], "d_text": ref["d_text"],
            "d_logit_scale": torch.tensor(ref["d_scale"], dtype=torch.float64)}
    bad = grad_problems(f"distill u={u:g}", got, want, 1.0)  # the reference already carries (g_c, g_d)
    assert not bad, "\n".join(bad)


def test_cyclip_seed_2_16(pkg):
    from test_gpu_cyclip import oracle as cyclip_oracle
    from dinosoft_b200.cyclip import CyCLIPLoss

    u, B, D, scale = 2.0 ** 16, 1000, 512, 50.0
    img, txt, _ = synth(31, B, D, 64)
    txt = torch.nn.functional.normalize(0.6 * img + 0.8 * txt, dim=-1).to(torch.bfloat16).float()
    ref = cyclip_oracle().loss_and_grads(img, txt, scale, 0.25, 0.5)
    im, tx = img.to(DEV).requires_grad_(True), txt.to(DEV).requires_grad_(True)
    sc = torch.tensor(scale, device=DEV, requires_grad=True)
    out = CyCLIPLoss(lambda_inmodal=0.25, lambda_crossmodal=0.5)(im, tx, sc, output_dict=True)
    (u * out["total_loss"]).backward()
    torch.cuda.synchronize()
    got = {"d_image": im.grad.double().cpu(), "d_text": tx.grad.double().cpu(), "d_logit_scale": sc.grad.double().cpu()}
    want = {"d_image": ref["d_image"], "d_text": ref["d_text"],
            "d_logit_scale": torch.tensor(ref["d_logit_scale"], dtype=torch.float64)}
    bad = grad_problems(f"cyclip u={u:g}", got, want, u)
    assert not bad, "\n".join(bad)


# --------------------------------------------------------------------------- (d) a real GradScaler step
def test_gradscaler_step_weighted(pkg, oracle):
    """The weighted configuration without a head, the way `--precision amp` runs it: forward under fp16 autocast,
    scaler.scale(total).backward(), unscale_, step, update.  The unscaled gradients meet the fp64 bar and no step is
    skipped (the scale stays at its initial 2^16)."""
    B, D, Dd, scale, seed, args = CONFIGS["weighted_sym_soft_mlp"]
    args = types.SimpleNamespace(**{**vars(args), "use_projection": False})
    img, txt, dino = synth(seed, B, D, Dd)
    im = img.to(DEV).requires_grad_(True)
    tx = txt.to(DEV).requires_grad_(True)
    sc = torch.tensor(scale, device=DEV, requires_grad=True)
    opt = torch.optim.SGD([im, tx, sc], lr=0.0)
    scaler = torch.amp.GradScaler("cuda")
    assert scaler.get_scale() == 2.0 ** 16
    loss = pkg.ClipLossWithDINOEnhancements()
    with torch.autocast("cuda", dtype=torch.float16):
        out = loss(im, tx, sc, dino.to(DEV), args, output_dict=True)
    scaler.scale(out["total_loss"]).backward()
    scaler.unscale_(opt)
    got = {"d_image": im.grad.double().cpu(), "d_text": tx.grad.double().cpu(), "d_logit_scale": sc.grad.double().cpu()}
    scaler.step(opt)
    scaler.update()
    r = oracle.loss_and_grads(img, txt, scale, dino, oracle_cfg(oracle, args), dtype=torch.float64)["ranks"][0]
    want = {"d_image": r["d_image"], "d_text": r["d_text"],
            "d_logit_scale": torch.tensor(r["d_logit_scale"], dtype=torch.float64)}
    bad = grad_problems("GradScaler fp16 autocast", got, want, 1.0)
    if scaler.get_scale() != 2.0 ** 16:
        bad.append(f"GradScaler: scale {scaler.get_scale():g} after update (a step was skipped)")
    assert not bad, "\n".join(bad)


# --------------------------------------------------------------------------- (e) CUDA-graph replay
@pytest.mark.parametrize("name", ["soft_text_mlp", "weighted_sym_soft_mlp"])
def test_graph_replay_follows_the_seed(pkg, name):
    """make_graphed, then backward of 2^16 x total and, in the next replay, of 2^15 x total (GradScaler's back-off):
    each equals u x the eager gradients of total_loss.  A captured backward that froze its seed fails this."""
    B, D, Dd, scale, seed, args = CONFIGS[name]
    loss = pkg.ClipLossWithDINOEnhancements()
    torch.manual_seed(5)
    loss.init_proj(D, Dd, DEV, "mlp")
    img, txt, dino = (t.to(DEV) for t in synth(seed, B, D, Dd))
    sc = torch.tensor(scale, device=DEV, requires_grad=True)
    img.requires_grad_(True)
    txt.requires_grad_(True)
    leaves = [img, txt, sc] + list(loss.image_to_dino_proj.parameters())

    def take_grads():
        out = [t.grad.detach().double().cpu() for t in leaves]
        for t in leaves:
            t.grad = None
        return out

    loss(img, txt, sc, dino, args, output_dict=True)["total_loss"].backward()
    eager = take_grads()
    step = pkg.make_graphed(loss, args, img, txt, sc, dino)
    for t in leaves:
        t.grad = None
    bad = []
    for u in (2.0 ** 16, 2.0 ** 15):
        total, _, _ = step(img, txt, sc, dino)
        (u * total).backward()
        for k, (g, e) in enumerate(zip(take_grads(), eager)):
            err = (g - u * e).abs().max().item() / max((u * e).abs().max().item(), 1e-300)
            print(f"[upstream] graphed {name} u={u:g} grad {k}: {err:.2e}")
            if not err < LIN_RTOL:
                bad.append(f"graphed {name} u={u:g} grad {k}: |g - u eager| / |u eager| = {err:.2e}")
    assert not bad, "\n".join(bad)
