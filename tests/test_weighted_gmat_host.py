"""Backward form of weighted plans (CPU, no GPU): `loss.GMAT = "never"` gives a weighted plan without DSOFT_F_GMAT
(the fused backward), `"auto"` and `"always"` keep the two-phase backward.  Runs the module against the
`OracleBackend` stand-in and records the flags of every plan it asks for."""
import types

import pytest
import torch

from oracle_backend import OracleBackend

F_GMAT, F_WEIGHTED = 16, 32


class _Recording(OracleBackend):
    def __init__(self, oracle):
        super().__init__(oracle)
        self.flags = []

    def plan(self, shape, device=None):
        self.flags.append(shape.flags)
        return super().plan(shape, device)


@pytest.mark.parametrize("mode,want_gmat", [("never", False), ("auto", True), ("always", True)])
def test_gmat_switch_for_weighted_plans(pkg, oracle, mode, want_gmat):
    from dinosoft_b200 import loss as loss_mod

    g = torch.Generator().manual_seed(1)
    b, D, Dd = 16, 16, 24
    img = torch.nn.functional.normalize(torch.randn(b, D, generator=g), dim=-1).requires_grad_(True)
    txt = torch.nn.functional.normalize(torch.randn(b, D, generator=g), dim=-1).requires_grad_(True)
    dino = torch.randn(b, Dd, generator=g)
    args = types.SimpleNamespace(use_projection=False, lambda_weighted=0.5, rho=0.2, c_clip=0.5,
                                 weight_text_symmetry=True)
    old = loss_mod.GMAT
    try:
        loss_mod.GMAT = mode
        m = pkg.ClipLossWithDINOEnhancements()
        be = _Recording(oracle)
        m._backend = be
        out = m(img, txt, torch.tensor(10.0), dino, args, output_dict=True)
        out["total_loss"].backward()
    finally:
        loss_mod.GMAT = old
        loss_mod._gmat_decisions.clear()
    weighted = [f for f in be.flags if f & F_WEIGHTED]
    assert weighted, be.flags
    assert all(bool(f & F_GMAT) == want_gmat for f in weighted), (mode, be.flags)
    assert torch.isfinite(img.grad).all() and torch.isfinite(txt.grad).all()
