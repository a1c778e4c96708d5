"""Host logic of the `weighted_scope` keyword (CPU, no GPU): argument checking and the reference's error order.
The default keeps the reference's failure of the lambda_weighted branch at world_size > 1 (pinned by
test_host_logic.py::test_error_behaviour_mirrors_reference)."""
import types

import pytest
import torch

from oracle_backend import OracleBackend


@pytest.mark.parametrize("bad", ["local", "GLOBAL", "", 1, True])
def test_bad_weighted_scope_raises(pkg, bad):
    with pytest.raises(ValueError, match="weighted_scope must be None or 'global'"):
        pkg.ClipLossWithDINOEnhancements(world_size=2, local_loss=True, weighted_scope=bad)


def test_weighted_scope_is_keyword_with_reference_default(pkg):
    import inspect

    sig = inspect.signature(pkg.ClipLossWithDINOEnhancements.__init__)
    assert sig.parameters["weighted_scope"].default is None
    assert pkg.ClipLossWithDINOEnhancements().weighted_scope is None
    assert pkg.ClipLossWithDINOEnhancements(weighted_scope="global").weighted_scope == "global"


def test_global_scope_still_needs_local_loss(pkg, oracle):
    """local_loss=False at world_size > 1 raises the reference's ValueError before anything else."""
    x = torch.nn.functional.normalize(torch.randn(8, 16), dim=-1)
    m = pkg.ClipLossWithDINOEnhancements(world_size=2, local_loss=False, weighted_scope="global")
    m._backend = OracleBackend(oracle)
    with pytest.raises(ValueError, match=r"Expected input batch_size \(16\) to match target batch_size \(8\)"):
        m(x, x, torch.tensor(10.0), torch.randn(8, 24),
          types.SimpleNamespace(lambda_weighted=0.5, use_projection=False), output_dict=True)


def test_row_blocks_compose_to_world1(oracle):
    """weighted_rows_ref.weighted_ce_global_rows: the mean over the row blocks is the oracle's weighted_ce of the
    concatenated batch, beta is the same on every block, and anything but the full [B, B] logits is refused."""
    from weighted_rows_ref import weighted_ce_global_rows

    g = torch.Generator().manual_seed(3)
    B, W = 48, 4
    b = B // W
    img = torch.nn.functional.normalize(torch.randn(B, 16, generator=g, dtype=torch.float64), dim=-1)
    txt = torch.nn.functional.normalize(img + 0.5 * torch.randn(B, 16, generator=g, dtype=torch.float64), dim=-1)
    dino = torch.randn(B, 24, generator=g, dtype=torch.float64)
    for sym in (False, True):
        cfg = oracle.OracleConfig(rho=0.2, c_clip=0.5, weight_text_symmetry=sym)
        li, lt = 20.0 * img @ txt.T, 20.0 * txt @ img.T
        one = oracle.weighted_ce(li, lt, dino, torch.arange(B), cfg)  # beta from fp32 row stds there, fp64 here
        parts = [weighted_ce_global_rows(li, lt, dino, slice(r * b, (r + 1) * b), 0.2, 0.5, sym) for r in range(W)]
        assert float(sum(p["loss"] for p in parts) / W) == pytest.approx(float(one["loss"]), rel=1e-6)
        for p in parts:
            assert p["beta_img"] == parts[0]["beta_img"] and p["beta_txt"] == parts[0]["beta_txt"]
            assert p["beta_img"] == pytest.approx(one["beta_img"], rel=1e-6)
            assert p["beta_txt"] == pytest.approx(one["beta_txt"], rel=1e-6)
        with pytest.raises(ValueError):
            weighted_ce_global_rows(li[:b], lt[:b], dino, slice(0, b), 0.2, 0.5, sym)


def test_rowblock_diagnostics_compose_to_world1():
    """weighted_rows_ref.weighted_ce_rows_branch with one block is weighted_ref.weighted_ce_branch, and the block
    means of the per-row diagnostics average to it."""
    import weighted_ref
    from weighted_rows_ref import weighted_ce_rows_branch

    g = torch.Generator().manual_seed(5)
    B, W = 40, 4
    b = B // W
    img = torch.nn.functional.normalize(torch.randn(B, 16, generator=g, dtype=torch.float64), dim=-1)
    txt = torch.nn.functional.normalize(img + 0.5 * torch.randn(B, 16, generator=g, dtype=torch.float64), dim=-1)
    dino = torch.randn(B, 24, generator=g, dtype=torch.float64)
    s = torch.tensor(20.0, dtype=torch.float64)
    for sym in (False, True):
        l1, d1 = weighted_ref.weighted_ce_branch(img, txt, s, dino, 0.2, 0.5, sym)
        lb, db = weighted_ce_rows_branch(img, txt, s, dino, 0.2, 0.5, sym, slice(0, B))
        assert float(lb) == pytest.approx(float(l1), rel=1e-12)
        for k in d1:
            assert float(db[k]) == pytest.approx(float(d1[k]), rel=1e-9, abs=1e-12), k
        parts = [weighted_ce_rows_branch(img, txt, s, dino, 0.2, 0.5, sym, slice(r * b, (r + 1) * b))
                 for r in range(W)]
        for k in ("pc_err_img", "l1_prob_shift_img", "corr_rhat_dprob_img", "ce_img_base", "ce_img_mod",
                  "delta_img_mean"):
            assert sum(float(p[1][k]) for p in parts) / W == pytest.approx(float(d1[k]), rel=1e-9), k
        assert float(sum(p[0] for p in parts) / W) == pytest.approx(float(l1), rel=1e-12)
