"""DistillClipLoss: drop-in for open_clip's ``DistillClipLoss`` (the ``--distill`` objective of ``create_loss``).

    x = s I T^T (student logits), t = s_t I_t T_t^T (teacher logits, ``dist_logit_scale`` already exp'd)
    contrastive = 1/2 [CE(x rows, diag) + CE(x columns, diag)]
    distill     = 1/2 [mean_i (lse(x_i.) - sum_j q_ij x_ij) + mean_j (lse(x_.j) - sum_i q_ij x_ij)]

with q the teacher's soft-max over rows (image -> text) or columns (text -> image): a cross-entropy against the
teacher's distribution, not a KL divergence, and no diagonal mask.  Upstream builds four [B, B] logit matrices and
their soft-maxes; here ``dsoft_distill_forward`` streams both products per tile and keeps per-row statistics only, and
``dsoft_distill_backward`` writes one fp16 logit-gradient matrix (both directions' terms, ``g_c`` and ``g_d`` kept
apart) for the two gradient GEMMs.  G takes 2 b B bytes and is only allocated in the backward.

Differences from upstream, deliberate:
  * the features are rounded to bf16 once and used as given (fp32 accumulation; s and s_t applied in fp32), as for
    the CLIP term of ``ClipLossWithDINOEnhancements``;
  * world_size > 1 needs ``local_loss=True``: rank r's rows are I_r T_all^T and T_r I_all^T for the student and the
    teacher, and its losses are the means over those rows.  One all-gather of the packed bf16 rows replaces
    ``gather_features``; the backward all-gathers the [4, b] row statistics when ``gather_with_grad`` is set;
  * gradients: features get the derivative of the sum of all ranks' losses with respect to this rank's rows (what
    ``gather_features`` with gradient delivers; without it the gathered copies are constants), ``logit_scale`` gets
    this rank's own losses.  This assumes the same s, s_t and upstream gradients on every rank, as under DDP.  The
    teacher gets no gradient: teacher inputs that require one while grad is enabled raise ``ValueError``.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _cabi
from .loss import _default_backend, _ptr, dist

__all__ = ["DistillClipLoss"]


def _pad8(x: torch.Tensor, width: int) -> torch.Tensor:
    return x if x.shape[1] == width else F.pad(x, (0, width - x.shape[1]))


class _DistillFn(torch.autograd.Function):
    """(image [b, D], text [b, D], logit_scale, teacher image [b, Dt], teacher text [b, Dt], dist_logit_scale)
    -> (contrastive, distill) of this rank (0-dim fp32 each)."""

    @staticmethod
    def forward(ctx, image, text, logit_scale, dist_image, dist_text, dist_logit_scale, world, rank, group,
                gather_with_grad):
        be = _default_backend(image.device)
        lib = be._lib
        dev = image.device
        b, D = image.shape
        Dt = dist_image.shape[1]
        Dp, Dtp = -(-D // 8) * 8, -(-Dt // 8) * 8  # zero columns change no dot product
        row_only = world > 1 and not gather_with_grad
        flags = _cabi.DSOFT_F_DISTILL | (_cabi.DSOFT_F_ROW_ONLY if row_only else 0)
        plan = be.plan(_cabi.Shape(b=b, world=world, rank=rank, D=Dp, Dp=Dtp, Dd=Dtp, flags=flags), dev)
        gathered = torch.empty((b * world, plan.row_elems), dtype=torch.bfloat16, device=dev)
        be.pack(plan, _pad8(image.detach(), Dp), _pad8(text.detach(), Dp), _pad8(dist_image.detach(), Dtp),
                _pad8(dist_text.detach(), Dtp), gathered)
        if world > 1:
            # the forward's only collective: one all-gather of the packed bf16 rows
            dist.all_gather_into_tensor(gathered.view(-1), gathered[rank * b:(rank + 1) * b].view(-1), group=group)
        state = torch.empty(plan.state_numel, dtype=torch.float32, device=dev)
        scratch = torch.empty(plan.fwd_scratch_numel, dtype=torch.float32, device=dev)
        stats = torch.empty((4, b), dtype=torch.float32, device=dev)
        losses = torch.empty(2, dtype=torch.float32, device=dev)
        ls = torch.as_tensor(logit_scale).detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        lt = torch.as_tensor(dist_logit_scale).detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        _cabi.check(lib.dsoft_distill_forward(plan.handle, _ptr(gathered), _ptr(ls), _ptr(lt), _ptr(state),
                                              _ptr(scratch), _ptr(stats), _ptr(losses), be._stream(gathered)),
                    "dsoft_distill_forward")
        ctx.save_for_backward(gathered, state, stats)
        ctx.plan = plan
        ctx.meta = (image.dtype, text.dtype, b, D, Dp, logit_scale.dtype, logit_scale.shape, world, group, row_only)
        return losses[0].clone(), losses[1].clone()

    @staticmethod
    def backward(ctx, g_contrastive, g_distill):
        gathered, state, stats = ctx.saved_tensors
        plan = ctx.plan
        idt, tdt, b, D, Dp, sdt, sshape, world, group, row_only = ctx.meta
        be = _default_backend(gathered.device)
        dev = gathered.device
        stats_all = stats
        if world > 1 and not row_only:
            stats_all = torch.empty((world, 4, b), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(stats_all.view(-1), stats.view(-1), group=group)
        scratch = torch.empty(plan.scratch_numel, dtype=torch.float32, device=dev)
        G = torch.empty(int(be._lib.dsoft_distill_g_bytes(plan.handle)) // 2, dtype=torch.float16, device=dev)
        d_image = torch.empty((b, Dp), dtype=torch.float32, device=dev)
        d_text = torch.empty((b, Dp), dtype=torch.float32, device=dev)
        d_scale = torch.empty(1, dtype=torch.float32, device=dev)
        gout = torch.stack([g_contrastive.detach().reshape(()), g_distill.detach().reshape(())]).to(torch.float32)
        _cabi.check(be._lib.dsoft_distill_backward(plan.handle, _ptr(gathered), _ptr(state), _ptr(scratch),
                                                   _ptr(stats_all), _ptr(G), _ptr(gout), _ptr(d_image), _ptr(d_text),
                                                   _ptr(d_scale), be._stream(gathered)),
                    "dsoft_distill_backward")
        return (d_image[:, :D].to(idt), d_text[:, :D].to(tdt), d_scale.reshape(sshape).to(sdt),
                None, None, None, None, None, None, None)


class DistillClipLoss(nn.Module):
    """Same constructor, forward signature and return values as upstream open_clip ``DistillClipLoss`` (2.31.0),
    plus ``process_group`` (the group the all-gathers run in; None: the default group)."""

    def __init__(self, local_loss: bool = False, gather_with_grad: bool = False, cache_labels: bool = False,
                 rank: int = 0, world_size: int = 1, use_horovod: bool = False, process_group=None):
        super().__init__()
        self.local_loss = local_loss
        self.gather_with_grad = gather_with_grad
        self.cache_labels = cache_labels
        self.rank = rank
        self.world_size = world_size
        self.use_horovod = use_horovod
        self.process_group = process_group
        # upstream keeps these for its label cache; the kernels index the positives directly
        self.prev_num_logits = 0
        self.labels = {}

    def forward(self, image_features, text_features, logit_scale, dist_image_features, dist_text_features,
                dist_logit_scale, output_dict: bool = False):
        if self.use_horovod:
            raise NotImplementedError("Horovod is not supported by the B200 path (NCCL only)")
        if self.world_size > 1 and not self.local_loss:
            # upstream evaluates the full [B, B] problem on every rank; the B200 path shards it by row blocks
            raise NotImplementedError("DistillClipLoss (B200 build) at world_size > 1 needs local_loss=True "
                                      "(--local-loss)")
        feats = (image_features, text_features, dist_image_features, dist_text_features)
        if any(f.dim() != 2 for f in feats) or image_features.shape != text_features.shape or \
                dist_image_features.shape != dist_text_features.shape or \
                dist_image_features.shape[0] != image_features.shape[0]:
            raise ValueError("features must be image / text [b, D] and teacher image / text [b, Dt]; got "
                             + ", ".join(str(tuple(f.shape)) for f in feats))
        if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad
                                           for t in (dist_image_features, dist_text_features, dist_logit_scale)):
            raise ValueError("DistillClipLoss gives the teacher no gradient: compute the teacher's features under "
                             "torch.no_grad() (as open_clip_train does) or detach them")
        dev = image_features.device
        if dev.type != "cuda" or any(f.device != dev for f in feats):
            raise RuntimeError("DistillClipLoss (B200 build) needs CUDA tensors on one sm_100 device; got "
                               + ", ".join(str(f.device) for f in feats) + ". There is no CPU fallback.")
        if self.world_size > 1 and dist is None:
            raise RuntimeError("DistillClipLoss at world_size > 1 needs torch.distributed")
        contrastive, distill = _DistillFn.apply(image_features, text_features, logit_scale, dist_image_features,
                                                dist_text_features, dist_logit_scale, self.world_size, self.rank,
                                                self.process_group, self.gather_with_grad)
        if output_dict:
            return {"contrastive_loss": contrastive, "distill_loss": distill}
        return contrastive, distill
