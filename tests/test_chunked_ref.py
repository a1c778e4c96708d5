"""The row-blocked fp64 checker used at full size (tests/chunked_ref.py) against the oracle, on the CPU."""
import pytest
import torch

from chunked_ref import chunked_reference
from gpu_util import make_args, oracle_cfg, synth


@pytest.mark.parametrize("use_head", [False, True])
@pytest.mark.parametrize("scale", [14.2857, 100.0])
def test_chunked_reference_matches_oracle(oracle, use_head, scale):
    B, D, Dd = 320, 64, 96
    img, txt, dino = synth(5, B, D, Dd)
    head = None
    if use_head:
        torch.manual_seed(1)
        H = (D + Dd) // 2
        l0, l1 = torch.nn.Linear(D, H), torch.nn.Linear(H, Dd)
        head = {"w0": l0.weight.detach(), "b0": l0.bias.detach(), "w1": l1.weight.detach(), "b1": l1.bias.detach()}
    args = make_args(use_projection=use_head)
    cfg = oracle_cfg(oracle, args, round_student_bf16=True)
    ref = oracle.loss_and_grads(img, txt, scale, dino, cfg, proj_params=head, dtype=torch.float64)["ranks"][0]
    blocks = [(0, 128), (128, 128), (256, 64)]
    got = chunked_reference(img, txt, dino, scale, head=head, blocks=blocks, slab=96)
    for k in ("classic_loss", "soft_loss", "total_loss"):
        assert got[k] == pytest.approx(ref[k], rel=1e-10), k
    assert got["d_logit_scale"] == pytest.approx(ref["d_logit_scale"], rel=1e-9)
    for blk in got["blocks"]:
        rows = slice(blk["row0"], blk["row0"] + blk["rows"])
        for k in ("d_image", "d_text", "d_student"):
            if blk[k] is None:
                continue
            want = ref[k][rows]
            err = (blk[k] - want).abs().max().item() / want.abs().max().item()
            assert err < 1e-9, (k, blk["row0"], err)


@pytest.mark.parametrize("sym", [False, True])
def test_chunked_weighted_loss_matches_oracle(oracle, sym):
    from chunked_ref import chunked_weighted_loss

    img, txt, dino = synth(3, 300, 32, 48)
    cfg = oracle.OracleConfig(lambda_weighted=0.5, rho=0.2, c_clip=0.5, weight_text_symmetry=sym)
    ref = oracle.loss_and_grads(img, txt, 30.0, dino, cfg)["ranks"][0]
    assert chunked_weighted_loss(img, txt, dino, 30.0, 0.2, 0.5, sym, slab=64) == pytest.approx(
        ref["weighted_loss"], rel=1e-9)


def test_chunked_reference_student_leaf(oracle):
    """student_values without a head: the student is a leaf, as in the oracle's rank_loss with a raw student."""
    from test_gpu_multirank import oracle_ranks

    B, D, Dd = 320, 64, 96
    img, txt, dino = synth(6, B, D, Dd)
    g = torch.Generator().manual_seed(2)
    student = (img @ torch.randn(D, Dd, generator=g)).to(torch.bfloat16).float()
    ref = oracle_ranks(oracle, img, txt, dino, student, 14.2857, 1, "global", False)[0]
    got = chunked_reference(img, txt, dino, 14.2857, blocks=[(0, 128), (192, 128)], slab=96, student_values=student)
    for k in ("classic_loss", "soft_loss", "total_loss"):
        assert got[k] == pytest.approx(float(ref["terms"][k]), rel=1e-10), k
    assert got["d_logit_scale"] == pytest.approx(ref["d_scale"], rel=1e-9)
    for blk in got["blocks"]:
        rows = slice(blk["row0"], blk["row0"] + blk["rows"])
        for k in ("d_image", "d_text", "d_student"):
            want = ref[k][rows]
            err = (blk[k] - want).abs().max().item() / want.abs().max().item()
            assert err < 1e-9, (k, blk["row0"], err)
