"""The loss under bf16 autocast (how train.py:285 and bench.py call it) against fp64, with the projection head on the
fused path: dsoft_head_forward for the head values and the head backward of _DinoSoftFn.backward.

The head kernel's own output (student columns, hidden activations) and the d_student the loss kernels return are
captured by wrapping CudaBackend.head_forward / backward.  Then
  * loss side: the oracle with the captured student as a leaf: loss terms 1e-4, d_text / d_logit_scale / d_student
    1e-3;
  * head side: tests/autocast_head_ref.py's backward from the oracle's d_student (on the kernel's hidden activations,
    themselves one bf16 rounding from the reference's): head-parameter gradients 1e-3 (L-inf and L2);
  * d_image = loss-side d_image + the head's dX: 1e-3, each element allowed one bf16 rounding of dX on top (the
    module adds the bf16 output of dh w1b, as autocast does).
World 1 at the BASELINE dims, ragged and config-4 dims, with the weighted branch and without the text term; the
bench's one-GPU size (B = 32768, where the head kernel walks all column tiles); NCCL at world 2 (shared soft tiles)
and 8 when the GPUs are there.  Both backward implementations."""
import os
import socket
import sys

import pytest
import torch

from conftest import ROOT
from autocast_head_ref import F64, assert_one_rounding, head_backward, linear_exact
from gpu_util import head_params_of, make_args, oracle_cfg, rel_err, synth

pytestmark = pytest.mark.gpu

LOSS_RTOL, GRAD_RTOL = 1e-4, 1e-3
GRAD_NAMES = {"dW1": "w0", "db1": "b0", "dW2": "w1", "db2": "b1"}  # reference key -> gpu_util.head_params_of key


@pytest.fixture(params=["two_phase", "fused"])
def gmat(request, pkg):
    """Both backward implementations (DSOFT_F_GMAT on / off)."""
    from dinosoft_b200 import loss as loss_mod

    old = loss_mod.GMAT
    loss_mod.GMAT = "always" if request.param == "two_phase" else "never"
    yield loss_mod.GMAT
    loss_mod.GMAT = old


def install_capture(setattr_fn=setattr):
    """Wrap CudaBackend.head_forward / backward; the returned dict receives the student columns and hidden activations
    the head kernel wrote (this rank's rows) and the finished d_student of the backward."""
    from dinosoft_b200.loss import CudaBackend

    got = {}
    head_forward_, backward_ = CudaBackend.head_forward, CudaBackend.backward

    def head_forward_capture(self, plan, gathered, w1, b1, w2, b2, hidden):
        head_forward_(self, plan, gathered, w1, b1, w2, b2, hidden)
        s = plan.shape
        got["student"] = gathered[s.rank * s.b:(s.rank + 1) * s.b, 2 * s.D:2 * s.D + s.Dp].clone()
        got["hidden"] = None if hidden is None else hidden.clone()

    def backward_capture(self, plan, gathered, state, scratch, lse_all, gout, lambdas, d_image, d_text, d_student,
                         d_scale, phase=0):
        backward_(self, plan, gathered, state, scratch, lse_all, gout, lambdas, d_image, d_text, d_student, d_scale,
                  phase=phase)
        if phase in (0, 2):  # the whole backward, or its last phase (shared soft tiles)
            got["d_student"] = d_student.clone()

    setattr_fn(CudaBackend, "head_forward", head_forward_capture)
    setattr_fn(CudaBackend, "backward", backward_capture)
    return got


def run_module(pkg, img, txt, dino, args, scale, setattr_fn=setattr, rank=0, world=1, **ctor):
    """One autocast forward + backward of this rank's rows; returns host copies of everything the checks need."""
    dev = torch.device("cuda", torch.cuda.current_device())
    got = install_capture(setattr_fn)
    loss = pkg.ClipLossWithDINOEnhancements(rank=rank, world_size=world, **ctor)
    torch.manual_seed(5)
    loss.init_proj(img.shape[1], dino.shape[1], dev, args.projection_type)
    im = img.detach().to(dev).clone().requires_grad_(True)
    tx = txt.detach().to(dev).clone().requires_grad_(True)
    sc = torch.tensor(scale, device=dev, requires_grad=True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = loss(im, tx, sc, dino.to(dev), args, output_dict=True)
    out["total_loss"].backward()
    torch.cuda.synchronize()
    assert "student" in got and "d_student" in got, "the head did not run on dsoft_head_forward"
    params = head_params_of(loss.image_to_dino_proj, args.projection_type)
    res = {k: float(out[k].detach()) for k in ("total_loss", "classic_loss", "soft_loss", "weighted_loss")}
    res.update(d_image=im.grad, d_text=tx.grad, d_scale=float(sc.grad),
               params={k: p.detach().clone() for k, p in params.items()},
               grads={k: p.grad.detach().clone() for k, p in params.items()},
               student=got["student"], hidden=got["hidden"], d_student=got["d_student"])
    return res


def check_grad(tag, name, got, want):
    linf, l2 = rel_err(got, want)
    print(f"[autocast head] {tag} {name}: linf={linf:.2e} l2={l2:.2e}")
    assert linf < GRAD_RTOL and l2 < GRAD_RTOL, (tag, name, linf, l2)


def check_d_image(tag, got, loss_side, dx_head):
    """d_image = loss side + the head's bf16 dX: 1e-3 of max |d_image| beyond one bf16 rounding of dX per element."""
    got, loss_side, dx_head = (t.detach().to(F64).cpu() for t in (got, loss_side, dx_head))
    want = loss_side + dx_head
    excess = ((got - want).abs() - 2.0 ** -8 * dx_head.abs()).clamp_min(0)
    linf = excess.max().item() / want.abs().max().item()
    l2 = (got - want).norm().item() / want.norm().item()
    print(f"[autocast head] {tag} d_image: linf beyond one dX rounding={linf:.2e} l2={l2:.2e}")
    assert linf < GRAD_RTOL and l2 < GRAD_RTOL, (tag, linf, l2)


def check_head(tag, res, x, d_student_ref):
    """The hidden activations of the run against the reference's forward, and its head-parameter gradients against
    the reference's backward from the fp64 d_student; returns the reference's dX.  The backward takes the kernel's
    hidden (one bf16 rounding from the reference's, checked here) as its operand: a pre-activation within the fp32
    accumulation error of zero may land on the other side of the ReLU, and one such row moves dW1 by far more than
    the rounding it comes from."""
    p = {k: v.to(x.device) for k, v in res["params"].items()}
    w1b = p["w0"].to(torch.bfloat16)
    w2b = p["w1"].to(torch.bfloat16) if "w1" in p else None
    hidden = None
    if w2b is not None:
        hidden = res["hidden"].to(x.device)
        assert_one_rounding(f"{tag} hidden", hidden, torch.relu(linear_exact(x, w1b, p["b0"])))
    ref = head_backward(x, w1b, w2b, hidden, d_student_ref.to(x.device))
    for key, name in GRAD_NAMES.items():
        if key in ref:
            check_grad(tag, name, res["grads"][name], ref[key])
    return ref["dX"]


def oracle_world1(oracle, args, img, txt, dino, student, scale):
    """Loss terms and gradients of the reference semantics (fp64), the student a leaf holding the captured values."""
    leaf = lambda t: t.detach().to(F64).cpu().clone().requires_grad_(True)
    im, tx, st = leaf(img), leaf(txt), leaf(student)
    sc = torch.tensor(float(scale), dtype=F64, requires_grad=True)
    out = oracle.rank_loss(im, tx, sc, dino.to(F64).cpu(), st, oracle_cfg(oracle, args))
    out["total_loss"].backward()
    return dict(terms={k: float(out[k].detach()) for k in ("total_loss", "classic_loss", "soft_loss", "weighted_loss")},
                d_image=im.grad, d_text=tx.grad, d_student=st.grad, d_scale=float(sc.grad))


WORLD1 = [
    # (B, D, Dd, projection type, extra args): MLP hidden width (D + Dd) / 2
    (256, 512, 768, "mlp", {}),                                  # config-1 dims
    (1000, 320, 208, "mlp", {}),                                 # ragged rows, Dp = 208, H = 264
    (1000, 320, 200, "linear", {}),                              # ragged rows, Dp = 200
    (384, 768, 1024, "mlp", {}),                                 # config-4 dims: both layers stream K > 512
    (512, 128, 192, "mlp", dict(lambda_weighted=0.5, rho=0.2, c_clip=0.5, weight_text_symmetry=False)),
    (512, 128, 192, "mlp", dict(lambda_weighted=0.5, rho=0.2, c_clip=0.5, weight_text_symmetry=True)),
    (512, 512, 768, "mlp", dict(soft_dino_to_text=False)),       # soft term without the text term
]


@pytest.mark.parametrize("B,D,Dd,ptype,extra", WORLD1,
                         ids=["c1", "ragged-mlp", "ragged-linear", "c4", "weighted", "weighted-sym", "no-text"])
def test_world1_against_fp64(pkg, oracle, gmat, monkeypatch, B, D, Dd, ptype, extra):
    img, txt, dino = synth(23, B, D, Dd)
    args = make_args(use_projection=True, projection_type=ptype, **extra)
    scale = 30.0
    res = run_module(pkg, img, txt, dino, args, scale, monkeypatch.setattr)
    tag = f"w1 B={B} {ptype} {extra} {gmat}"
    want = oracle_world1(oracle, args, img, txt, dino, res["student"].float(), scale)
    keys = ("total_loss", "classic_loss", "soft_loss") + (("weighted_loss",) if extra.get("lambda_weighted") else ())
    for k in keys:
        print(f"[autocast head] {tag} {k}: got={res[k]:.7f} ref={want['terms'][k]:.7f}")
        assert res[k] == pytest.approx(want["terms"][k], rel=LOSS_RTOL, abs=1e-5), (tag, k)
    assert res["d_scale"] == pytest.approx(want["d_scale"], rel=GRAD_RTOL, abs=1e-7), tag
    check_grad(tag, "d_text", res["d_text"], want["d_text"])
    check_grad(tag, "d_student", res["d_student"], want["d_student"])
    x = img.to(torch.bfloat16)
    dx = check_head(tag, res, x, want["d_student"])
    check_d_image(tag, res["d_image"], want["d_image"], dx)


def test_full_size_against_fp64(pkg, gmat, monkeypatch):
    """The bench's one-GPU line (B = 32768, D = 512, Dd = 768, MLP head; the head kernel walks all column tiles):
    head values on every row, losses and three sampled 128-row blocks against the row-blocked fp64 reference, head
    gradients from the captured d_student of all rows."""
    from chunked_ref import chunked_reference

    B, D, Dd, scale = 32768, 512, 768, 14.2857
    img, txt, dino = synth(77, B, D, Dd, device="cuda")
    args = make_args(use_projection=True)
    res = run_module(pkg, img, txt, dino, args, scale, monkeypatch.setattr)
    tag = f"B={B} {gmat}"
    x = img.to(torch.bfloat16)
    p = res["params"]
    w1b, w2b = p["w0"].to(torch.bfloat16), p["w1"].to(torch.bfloat16)
    assert_one_rounding(f"{tag} hidden", res["hidden"], torch.relu(linear_exact(x, w1b, p["b0"])))
    assert_one_rounding(f"{tag} student", res["student"], linear_exact(res["hidden"], w2b, p["b1"]))
    # head gradients from the d_student the loss kernels returned (all rows)
    h = res["hidden"]
    ref = head_backward(x, w1b, w2b, h, res["d_student"])
    for key, name in GRAD_NAMES.items():
        check_grad(tag, name, res["grads"][name], ref[key])
    blocks = [(0, 128), (B // 2 + 128, 128), (B - 128, 128)]
    want = chunked_reference(img, txt, dino, scale, blocks=blocks, lambdas=(1.0, 0.5, 0.5), teacher_temp=0.15,
                             text_temp=0.02, slab=2048, student_values=res["student"])
    for k in ("total_loss", "classic_loss", "soft_loss"):
        print(f"[autocast head] {tag} {k}: got={res[k]:.7f} ref={want[k]:.7f}")
        assert res[k] == pytest.approx(want[k], rel=LOSS_RTOL), k
    assert res["d_scale"] == pytest.approx(want["d_logit_scale"], rel=GRAD_RTOL, abs=1e-7)
    for blk in want["blocks"]:
        rows = slice(blk["row0"], blk["row0"] + blk["rows"])
        btag = f"{tag} rows {blk['row0']}.."
        check_grad(btag, "d_text", res["d_text"][rows], blk["d_text"])
        check_grad(btag, "d_student", res["d_student"][rows], blk["d_student"])
        dx = head_backward(x[rows], w1b, w2b, h[rows], blk["d_student"])["dX"]
        check_d_image(btag, res["d_image"][rows], blk["d_image"], dx)


# ---- NCCL, one process per GPU (the test_gpu_dist pattern)
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, B, D, Dd, scale, gmat, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["DSOFT_GMAT"] = gmat  # backward implementation (read when the package is imported)
    os.environ["DSOFT_SYM_W"] = "1"  # share the symmetric soft tiles across ranks wherever the plan allows it
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import dinosoft_b200 as pkg

    img, txt, dino = synth(21, B, D, Dd)
    b = B // world
    rows = slice(rank * b, (rank + 1) * b)
    res = run_module(pkg, img[rows], txt[rows], dino[rows], make_args(use_projection=True), scale, rank=rank,
                     world=world, local_loss=True, gather_with_grad=True, soft_scope="global")
    ret[rank] = {k: (v.cpu() if torch.is_tensor(v) else {n: t.cpu() for n, t in v.items()} if isinstance(v, dict)
                     else v) for k, v in res.items()}
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("gmat_env", ["always", "never"], ids=["two_phase", "fused"])
@pytest.mark.parametrize("world,B,D,Dd", [(2, 1024, 512, 768), (8, 4096, 128, 192)], ids=["w2-symw", "w8"])
def test_nccl_every_rank(oracle, world, B, D, Dd, gmat_env):
    """Every rank's losses and gradients, and - per rank, on its own rows - the head-parameter gradients."""
    import torch.multiprocessing as mp
    from test_gpu_multirank import oracle_ranks

    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    scale = 30.0
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), B, D, Dd, scale, gmat_env, ret), nprocs=world, join=True)
    img, txt, dino = synth(21, B, D, Dd)
    b = B // world
    student = torch.cat([ret[r]["student"].float() for r in range(world)])  # the operand the kernels used
    want = oracle_ranks(oracle, img, txt, dino, student, scale, world, "global", True)
    for r in range(world):
        res, ref = ret[r], want[r]
        tag = f"rank {r} of {world} {gmat_env}"
        for k in ("total_loss", "classic_loss", "soft_loss"):
            assert res[k] == pytest.approx(float(ref["terms"][k]), rel=LOSS_RTOL, abs=1e-5), (tag, k)
        assert res["d_scale"] == pytest.approx(ref["d_scale"], rel=GRAD_RTOL, abs=1e-7), tag
        check_grad(tag, "d_text", res["d_text"], ref["d_text"])
        check_grad(tag, "d_student", res["d_student"], ref["d_student"])
        x = img[r * b:(r + 1) * b].to(torch.bfloat16)
        dx = check_head(tag, res, x, ref["d_student"])
        check_d_image(tag, res["d_image"], ref["d_image"], dx)
