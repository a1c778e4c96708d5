"""fp64 reference of the projection head as the loss runs it under bf16 autocast (train.py:285): TEST INFRASTRUCTURE.

A Linear or Linear-ReLU-Linear head (loss.py:214-238) with bf16 weights and input, fp32 biases.  The values are
rounded to bf16 where autocast rounds them - every nn.Linear output and the gradient entering a bf16 output - and
everything else is exact (fp64):

    h      = bf16(relu(x w1b^T + b1))          dz  = bf16(d_student)
    z      = bf16(h w2b^T + b2)                dW2 = dz^T h           db2 = sum(d_student)
                                               dh  = bf16(dz w2b) * [h > 0]
                                               dW1 = dh^T x           db1 = sum(dh)
                                               dX  = bf16(dh w1b)

The Linear head is the last layer alone: z = bf16(x w1b^T + b1), dW1 = dz^T x, db1 = sum(d_student),
dX = bf16(dz w1b).  A bias may be None.

Two places where the module deliberately differs from torch.autocast, both towards the exact value (and which the
host test pins against torch.autocast): the biases stay fp32 in the forward (autocast rounds them to bf16 first),
and the parameter gradients are not rounded to bf16 (autocast returns bf16 gradients of the bf16 weight copies;
db2 then even sums the bf16 dz, where the module sums the fp32 d_student)."""
from __future__ import annotations

import torch

F64 = torch.float64


def bf16(t: torch.Tensor) -> torch.Tensor:
    """Round to bf16 and back to the dtype of `t`."""
    return t.to(torch.bfloat16).to(t.dtype)


def linear_exact(x, w, bias=None):
    """x w^T + bias in fp64, before the bf16 rounding of the output (one nn.Linear under autocast)."""
    y = x.to(F64) @ w.to(F64).T
    return y if bias is None else y + bias.to(F64)


def head_forward(x, w1b, b1, w2b=None, b2=None):
    """(h, z) in fp64 with the bf16 values autocast gives; h is None for the Linear head."""
    if w2b is None:
        return None, bf16(linear_exact(x, w1b, b1))
    h = bf16(torch.relu(linear_exact(x, w1b, b1)))
    return h, bf16(linear_exact(h, w2b, b2))


def head_backward(x, w1b, w2b, h, d_student):
    """Gradients of the head (fp64) for the upstream gradient d_student of its output.  Keys: dW1, db1 (first or only
    layer), dW2, db2 (second layer of the MLP), dX (the head's share of d_image)."""
    x, w1b = x.to(F64), w1b.to(F64)
    ds = d_student.to(F64)
    dz = bf16(ds)
    if w2b is None:
        return dict(dW1=dz.T @ x, db1=ds.sum(0), dX=bf16(dz @ w1b))
    h = h.to(F64)
    dh = bf16(dz @ w2b.to(F64)) * (h > 0)
    return dict(dW1=dh.T @ x, db1=dh.sum(0), dW2=dz.T @ h, db2=ds.sum(0), dX=bf16(dh @ w1b))


def assert_one_rounding(name, got, exact, mean_rtol=2e-3):
    """`got` (bf16 output of a kernel) is bf16(exact) up to the fp32 accumulation: within one bf16 rounding (2^-8
    relative) plus a tiny floor for values next to zero everywhere, and on average well inside that bound."""
    got, exact = got.to(F64), exact.to(F64)
    err = (got - exact).abs()
    floor = 2.0 ** -14 * exact.abs().max().item()
    bad = err > 2.0 ** -8 * exact.abs() + floor
    assert not bool(bad.any()), (name, int(bad.sum()), err.max().item())
    mean = err.mean().item() / exact.abs().mean().item()
    print(f"[head] {name}: max err {err.max().item():.2e}, mean err / mean |ref| {mean:.2e}")
    assert mean < mean_rtol, (name, mean)
