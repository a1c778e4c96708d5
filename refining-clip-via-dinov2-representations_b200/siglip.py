"""SigLIP loss: drop-in for open_clip's ``SigLipLoss`` (the ``--siglip`` objective of ``create_loss``).

    z_ij = s <I_i, T_j> + beta,   l_ij = +1 if j is i's own caption (global index), -1 otherwise
    L_r  = (1/b) sum_{i in rank r's rows} sum_{j < B} softplus(-l_ij z_ij)     (= -logsigmoid(labels * logits).sum() / b
                                                                                over the local and all neighbour blocks)

Every pair's gradient depends only on that pair's logit, so the forward tile kernel (``dsoft_siglip_forward``) writes
the fp16 logit-gradient matrix G while it computes the loss, and the backward is the two gradient GEMMs
(``dsoft_siglip_backward``).  Nothing of size B x B exists in fp32; G takes 2 b B bytes per direction (the text rows'
G at world > 1 is computed in the backward) and is only allocated when a gradient is wanted.

Differences from upstream, deliberate:
  * the features are rounded to bf16 once and used as given (fp32 accumulation; s and beta applied in fp32), as for
    the CLIP term of ``ClipLossWithDINOEnhancements``;
  * at world_size > 1 one all-gather of the packed bf16 rows replaces the neighbour exchange: ``dist_impl`` is
    validated as upstream does and otherwise ignored (every implementation gives the same loss);
  * gradients: features get the derivative of the sum of all ranks' losses with respect to this rank's rows (what
    upstream's exchange with gradient delivers), ``logit_scale`` / ``logit_bias`` get this rank's own loss.  This
    assumes the same s, beta and upstream gradient on every rank, as under DDP.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _cabi
from .loss import _default_backend, _ptr, dist

__all__ = ["SigLipLoss"]

DIST_IMPLS = ("bidir", "shift", "reduce", "gather")


class _SigLipFn(torch.autograd.Function):
    """(image [b, D], text [b, D], logit_scale, logit_bias or None) -> this rank's loss (0-dim fp32)."""

    @staticmethod
    def forward(ctx, image, text, logit_scale, logit_bias, world, rank, group):
        be = _default_backend(image.device)
        lib = be._lib
        dev = image.device
        b, D = image.shape
        Dp = -(-D // 8) * 8  # the packed rows need a multiple of 8; zero columns change no dot product
        img, txt = image.detach(), text.detach()
        if Dp != D:
            img, txt = F.pad(img, (0, Dp - D)), F.pad(txt, (0, Dp - D))
        plan = be.plan(_cabi.Shape(b=b, world=world, rank=rank, D=Dp, Dp=0, Dd=0, flags=_cabi.DSOFT_F_SIGLIP), dev)
        gathered = torch.empty((b * world, plan.row_elems), dtype=torch.bfloat16, device=dev)
        be.pack(plan, img, txt, None, None, gathered)
        if world > 1:
            # the only collective: one all-gather of the packed bf16 rows (image | text)
            dist.all_gather_into_tensor(gathered.view(-1), gathered[rank * b:(rank + 1) * b].view(-1), group=group)
        state = torch.empty(plan.state_numel, dtype=torch.float32, device=dev)
        scratch = torch.empty(plan.fwd_scratch_numel, dtype=torch.float32, device=dev)
        G = None
        if any(ctx.needs_input_grad[:4]):
            G = torch.empty(int(lib.dsoft_siglip_g_bytes(plan.handle)) // 2, dtype=torch.float16, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        ls = logit_scale.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        lb = None if logit_bias is None else logit_bias.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        _cabi.check(lib.dsoft_siglip_forward(plan.handle, _ptr(gathered), _ptr(ls), _ptr(lb), _ptr(state),
                                             _ptr(scratch), _ptr(G), _ptr(loss), be._stream(gathered)),
                    "dsoft_siglip_forward")
        ctx.save_for_backward(gathered, state, G)
        ctx.plan = plan
        ctx.meta = (image.dtype, text.dtype, b, D, Dp, logit_scale.dtype, logit_scale.shape,
                    None if logit_bias is None else (logit_bias.dtype, logit_bias.shape))
        return loss.reshape(())

    @staticmethod
    def backward(ctx, gloss):
        gathered, state, G = ctx.saved_tensors
        plan = ctx.plan
        idt, tdt, b, D, Dp, sdt, sshape, bmeta = ctx.meta
        be = _default_backend(gathered.device)
        dev = gathered.device
        scratch = torch.empty(plan.scratch_numel, dtype=torch.float32, device=dev)
        d_image = torch.empty((b, Dp), dtype=torch.float32, device=dev)
        d_text = torch.empty((b, Dp), dtype=torch.float32, device=dev)
        d_scale = torch.empty(1, dtype=torch.float32, device=dev)
        d_bias = torch.empty(1, dtype=torch.float32, device=dev) if bmeta is not None else None
        gout = gloss.detach().to(torch.float32).reshape(1).contiguous()
        _cabi.check(be._lib.dsoft_siglip_backward(plan.handle, _ptr(gathered), _ptr(state), _ptr(scratch), _ptr(G),
                                                  _ptr(gout), _ptr(d_image), _ptr(d_text), _ptr(d_scale),
                                                  _ptr(d_bias), be._stream(gathered)),
                    "dsoft_siglip_backward")
        g_bias = None if d_bias is None else d_bias.reshape(bmeta[1]).to(bmeta[0])
        return (d_image[:, :D].to(idt), d_text[:, :D].to(tdt), d_scale.reshape(sshape).to(sdt), g_bias,
                None, None, None)


class SigLipLoss(nn.Module):
    """Same constructor, forward signature and return values as upstream open_clip ``SigLipLoss`` (2.31.0), plus
    ``process_group`` (the group the all-gather runs in; None: the default group)."""

    def __init__(self, cache_labels: bool = False, rank: int = 0, world_size: int = 1,
                 dist_impl: Optional[str] = None, process_group=None):
        super().__init__()
        self.cache_labels = cache_labels
        self.rank = rank
        self.world_size = world_size
        self.dist_impl = dist_impl or "bidir"
        assert self.dist_impl in DIST_IMPLS
        self.process_group = process_group
        # upstream keeps these for a label cache it does not use
        self.prev_num_logits = 0
        self.labels = {}

    def forward(self, image_features, text_features, logit_scale, logit_bias=None, output_dict: bool = False):
        if image_features.dim() != 2 or image_features.shape != text_features.shape:
            raise ValueError(f"image and text features must both be [b, D]; got {tuple(image_features.shape)} and "
                             f"{tuple(text_features.shape)}")
        if image_features.device.type != "cuda" or text_features.device != image_features.device:
            raise RuntimeError("SigLipLoss (B200 build) needs CUDA tensors on one sm_100 device; got "
                               f"{image_features.device} and {text_features.device}. There is no CPU fallback.")
        if self.world_size > 1 and dist is None:
            raise RuntimeError("SigLipLoss at world_size > 1 needs torch.distributed")
        loss = _SigLipFn.apply(image_features, text_features, logit_scale, logit_bias, self.world_size, self.rank,
                               self.process_group)
        return {"contrastive_loss": loss} if output_dict else loss
