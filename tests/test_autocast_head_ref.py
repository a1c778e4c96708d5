"""tests/autocast_head_ref.py against torch.autocast itself (CPU, bf16): the reference's rounding points are the ones
autocast uses for nn.Linear / ReLU, forward and backward, so the GPU tests that compare the fused head with it
measure the kernels and not a guess about autocast."""
import pytest
import torch

from autocast_head_ref import F64, bf16, head_backward, head_forward

BF = torch.bfloat16


def bf16_step(t):
    """Spacing of bf16 numbers at |t| (one rounding step)."""
    return torch.exp2(torch.floor(torch.log2(t.abs().clamp_min(1e-30))) - 7)


def assert_within_one_step(name, got, want, max_frac=0.02):
    """Equal as bf16 numbers except on isolated elements, which may be one step apart (fp32 sums in a different
    order land on the other side of a rounding boundary); L2 below 1e-3."""
    got, want = got.detach().to(F64), want.detach().to(F64)
    diff = (got - want).abs()
    step = bf16_step(torch.maximum(got.abs(), want.abs()))
    frac = (diff > 0).double().mean().item()
    l2 = (diff.norm() / want.norm().clamp_min(1e-30)).item()
    print(f"[autocast ref] {name}: {frac:.2%} of elements differ, l2={l2:.1e}")
    assert bool((diff <= step * (1 + 1e-6)).all()), (name, (diff / step).max().item())
    assert frac <= max_frac, (name, frac)
    assert l2 < 1e-3, (name, l2)


@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("ptype", ["mlp", "linear"])
@pytest.mark.parametrize("b,D,H,Dp", [(37, 24, 40, 56), (300, 72, 104, 136)])
def test_reference_matches_cpu_autocast(ptype, bias, b, D, H, Dp):
    g = torch.Generator().manual_seed(b + D)
    torch.manual_seed(b)
    if ptype == "mlp":
        head = torch.nn.Sequential(torch.nn.Linear(D, H, bias=bias), torch.nn.ReLU(), torch.nn.Linear(H, Dp, bias=bias))
        lin = [head[0], head[2]]
    else:
        head = torch.nn.Linear(D, Dp, bias=bias)
        lin = [head]
    with torch.no_grad():
        # autocast rounds the fp32 biases to bf16 before adding them, the fused head adds them in fp32: with
        # bf16-representable biases both sums are the same, and the comparison is about the rounding points alone
        for p in head.parameters():
            p.copy_(bf16(p))
    x = torch.nn.functional.normalize(torch.randn(b, D, generator=g), dim=-1).to(BF).float().requires_grad_(True)
    d_student = 1e-3 * torch.randn(b, Dp, generator=g)  # fp32, not bf16-representable: dz is a rounding point
    grabbed = {}
    if ptype == "mlp":
        head[1].register_forward_hook(lambda m, i, o: grabbed.__setitem__("h", o.detach()))
    with torch.autocast("cpu", dtype=BF):
        z = head(x)
    assert z.dtype == BF
    z.backward(d_student.to(z.dtype))

    w1b = lin[0].weight.detach().to(BF)
    w2b = lin[1].weight.detach().to(BF) if ptype == "mlp" else None
    bias_of = lambda m: None if m.bias is None else m.bias.detach()
    h, z_ref = head_forward(x.detach().to(BF), w1b, bias_of(lin[0]), w2b, bias_of(lin[1]) if w2b is not None else None)
    assert_within_one_step("z", z, z_ref)
    if h is not None:
        assert_within_one_step("h", grabbed["h"], h)
    ref = head_backward(x.detach().to(BF), w1b, w2b, h, d_student)
    assert_within_one_step("dX", x.grad, ref["dX"])
    # autocast hands back bf16 parameter gradients (of the bf16 weight copies); the reference keeps them exact
    assert_within_one_step("dW1", lin[0].weight.grad, bf16(ref["dW1"]))
    if w2b is not None:
        assert_within_one_step("dW2", lin[1].weight.grad, bf16(ref["dW2"]))
    if bias:
        last = lin[-1]
        # the bias of the last layer: autocast sums the bf16 dz, the module (and the reference) the fp32 d_student
        dz = bf16(d_student.to(F64))
        assert_within_one_step("db(last)", last.bias.grad, bf16(dz.sum(0)))
        assert torch.equal(ref["db2" if w2b is not None else "db1"], d_student.to(F64).sum(0))
        if w2b is not None:
            assert_within_one_step("db1", lin[0].bias.grad, bf16(ref["db1"]))
