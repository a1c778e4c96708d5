"""Drop-in replacement for the reference's DINO-Soft loss module, backed by hand-written sm_100a CUDA.

Mirrors (names, argument meaning, return values, error behaviour) the reference's
``src/open_clip/loss.py``:

    gather_features .................... loss.py:23-81
    compute_student_tau ................ loss.py:166-175
    ClipLossWithDINOEnhancements ....... loss.py:190-607   (constructed by factory.py:566-576,
                                                            called from open_clip_train/train.py:344-351)

The B x B work (CLIP logits + CE, teacher/student/text Gram matrices, soft-max, KL, and the whole
backward) runs in ``libdsoft.so`` through the C ABI in ``include/dsoft.h``; PyTorch is used for device
memory, streams, the NCCL all-gather and the tiny projection head (loss.py:214-238), nothing else.
There is no CPU path and no PyTorch fallback for the kernels: a non-CUDA input raises.

Differences from the reference that are deliberate and documented in DESIGN.md:
  * operands of the tensor-core products are bf16 (features are rounded once; the projection-head output
    is rounded with a straight-through gradient); all soft-max / KL arithmetic is fp32;
  * at world_size > 1 the soft terms default to the *global* row block (``soft_scope="global"``);
    ``soft_scope="local"`` reproduces the reference's local b x b block;
  * the weighted-CE branch (loss.py:416-471, lambda_weighted > 0, off by default) runs in the same fused kernels
    (fp32 logits also under autocast, beta kept on the device instead of `.item()`).  The reference only runs it on
    one rank; at world_size > 1 it raises like the reference unless ``weighted_scope="global"``, which gives rank r
    the rows [r b, (r+1) b) of the branch on the concatenated batch (beta from the row stds of all B rows);
  * Horovod is not supported (``use_horovod=True`` raises).
"""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd.function import once_differentiable

try:  # same guard as the reference (loss.py:7-13)
    import torch.distributed.nn  # noqa: F401
    from torch import distributed as dist

    has_distributed = True
except ImportError:  # pragma: no cover
    dist = None
    has_distributed = False

from . import _cabi
from .feature_store import DinoRows

__all__ = [
    "gather_features",
    "compute_student_tau",
    "ClipLossWithDINOEnhancements",
    "CudaBackend",
]


# --------------------------------------------------------------------------------------------------
# gather_features (loss.py:23-81) - NCCL / torch.distributed only
# --------------------------------------------------------------------------------------------------
def gather_features(
    image_features,
    text_features,
    local_loss=False,
    gather_with_grad=False,
    rank=0,
    world_size=1,
    use_horovod=False,
):
    """Same contract as the reference's ``gather_features``; used by ``get_logits`` (API parity only -
    the fused loss path gathers one packed bf16 buffer instead, see ``_DinoSoftFn``)."""
    assert has_distributed, "torch.distributed did not import correctly, please use a PyTorch version with support."
    if use_horovod:
        raise NotImplementedError("Horovod is not supported by the B200 DINO-Soft path (NCCL only)")
    if gather_with_grad:
        all_image_features = torch.cat(torch.distributed.nn.all_gather(image_features), dim=0)
        all_text_features = torch.cat(torch.distributed.nn.all_gather(text_features), dim=0)
    else:
        gathered_image_features = [torch.zeros_like(image_features) for _ in range(world_size)]
        gathered_text_features = [torch.zeros_like(text_features) for _ in range(world_size)]
        dist.all_gather(gathered_image_features, image_features)
        dist.all_gather(gathered_text_features, text_features)
        if not local_loss:
            gathered_image_features[rank] = image_features
            gathered_text_features[rank] = text_features
        all_image_features = torch.cat(gathered_image_features, dim=0)
        all_text_features = torch.cat(gathered_text_features, dim=0)
    return all_image_features, all_text_features


def compute_student_tau(logit_scale_tensor):
    """loss.py:166-175 (host-visible twin of the device computation in prep_scalars_kernel)."""
    val = logit_scale_tensor.detach()
    scale_mult = torch.where(val > 10, val, val.exp())
    scale_mult = torch.clamp(scale_mult, max=100)
    return (1.0 / scale_mult).clamp(min=0.008, max=0.02)


# --------------------------------------------------------------------------------------------------
# C-ABI backend
# --------------------------------------------------------------------------------------------------
_DTYPES = {torch.float32: _cabi.DT_F32, torch.bfloat16: _cabi.DT_BF16, torch.float16: _cabi.DT_F16}


class _Plan:
    __slots__ = ("handle", "row_elems", "state_numel", "scratch_numel", "fwd_scratch_numel", "flops",
                 "launches_fwd", "launches_bwd", "shape", "dino_col", "symw", "lse_rows", "wsig")


class _SymW:
    """Exchange layout of a plan that shares the symmetric soft tiles across ranks (dsoft_plan_symw_info).

    Primed block k (columns [k b, (k+1) b) relative to this rank's first row) holds what this rank computed for the
    rows of rank (rank + k) % W; the last block may be half a block (see include/dsoft.h)."""

    def __init__(self, info, W, rank):
        (_, self.b, self.Bcol, self.off_colsum, self.ncols, self.off_r3, self.Dz, self.off_r4, self.Dx, self.off_a3,
         self.off_a4, self.nsplit) = [int(x) for x in info]
        self.W, self.rank = W, rank
        b = self.b
        # (peer, primed block, rows) this rank sends / receives
        self.sends = [((rank + k) % W, k, min(b, self.ncols - k * b)) for k in range(1, -(-self.ncols // b))]
        self.recvs = []
        for k in range(1, W):
            s = (rank - k) % W
            if W % 2:
                rows = b if k <= (W - 1) // 2 else 0
            elif k < W // 2:
                rows = b
            elif k == W // 2:
                rows = b if s < W // 2 else b // 2  # the contested block: see the plan's ownership rule
            else:
                rows = 0
            if rows:
                self.recvs.append((s, k, rows))

    # ---- views into the scratch buffers
    def colsum(self, fwd_scratch):
        return fwd_scratch[self.off_colsum:self.off_colsum + 6 * self.Bcol].view(6, self.Bcol)

    def remote(self, scratch, which):
        off, d = (self.off_r3, self.Dz) if which == 0 else (self.off_r4, self.Dx)
        n = self.ncols - self.b
        return scratch[off:off + n * d].view(n, d)

    def own(self, scratch, which):
        off, d = (self.off_a3, self.Dz) if which == 0 else (self.off_a4, self.Dx)
        return scratch[off:off + self.b * d].view(self.b, d)

    # ---- phase schedule.  The soft part (phase 1) and its exchange form one chain, the CLIP part (phase 3) is
    # independent of both: the chain runs on a high-priority second stream and the CLIP part on the caller's, so the
    # block scheduler places the soft CTAs first, CLIP CTAs fill the partial waves, and what is left of the CLIP part
    # runs beside the exchange (2 GPUs, global batch 32768: 7.36 ms per step against 7.86 ms with everything in
    # line).  While the kernel recorder is on (bench.py's per-kernel pass) everything stays on the caller's stream.
    _side = {}

    def run(self, dev, concurrency, call, exchange):
        """call(phase) issues one phase of the C pass on the current stream; exchange() the collective after 1."""
        call(4)
        if dev.type != "cuda" or concurrency == 2:
            call(1)
            exchange()
            call(3)
            call(2)
            return
        side = _SymW._side.get(dev.index)
        if side is None:
            side = _SymW._side[dev.index] = torch.cuda.Stream(dev, priority=-1)
        main = torch.cuda.current_stream(dev)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            call(1)
            exchange()
        call(3)
        main.wait_stream(side)
        call(2)

    # ---- the two exchanges over NCCL
    def exchange_forward(self, fwd_scratch, group):
        cs = self.colsum(fwd_scratch)
        send = torch.zeros((self.W, 6, self.b), dtype=torch.float32, device=cs.device)
        for peer, k, rows in self.sends:
            send[peer, :, :rows] = cs[:, k * self.b:k * self.b + rows]
        recv = torch.empty_like(send)
        dist.all_to_all_single(recv, send, group=group)
        cs[:, :self.b] += recv.sum(0)

    def exchange_backward(self, scratch, group):
        ops, landed = [], []
        for which in ((0, 1) if self.Dx else (0,)):
            rem, own = self.remote(scratch, which), self.own(scratch, which)
            for peer, k, rows in self.sends:
                # peers are ranks WITHIN the loss's process group (the module's `rank` / `world_size`)
                ops.append(dist.P2POp(dist.isend, rem[(k - 1) * self.b:(k - 1) * self.b + rows], group=group,
                                      group_peer=peer))
            for peer, k, rows in self.recvs:
                buf = torch.empty((rows, rem.shape[1]), dtype=torch.float32, device=rem.device)
                ops.append(dist.P2POp(dist.irecv, buf, group=group, group_peer=peer))
                landed.append((own, rows, buf))
        for req in dist.batch_isend_irecv(ops):
            req.wait()
        for own, rows, buf in landed:
            own[:rows] += buf


def _rowmajor(x: torch.Tensor) -> torch.Tensor:
    if x.dtype not in _DTYPES:
        x = x.float()
    if x.dim() != 2 or x.stride(1) != 1:
        x = x.contiguous()
    return x


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


class CudaBackend:
    """Calls libdsoft.so.  One plan per problem shape, cached for the life of the process."""

    name = "sm100a-cabi"

    def __init__(self):
        self._lib = _cabi.lib()
        self._plans = {}

    def plan(self, shape: "_cabi.Shape", device: Optional[torch.device] = None) -> _Plan:
        if device is not None and device.index is not None and torch.cuda.current_device() != device.index:
            torch.cuda.set_device(device)
        key = (shape.key(), torch.cuda.current_device())
        p = self._plans.get(key)
        if p is None:
            import ctypes as C

            h = C.c_void_p()
            _cabi.check(self._lib.dsoft_plan_create(C.byref(shape), C.byref(h)), "dsoft_plan_create")
            p = _Plan()
            p.handle = h
            p.row_elems = int(self._lib.dsoft_plan_gathered_row_elems(h))
            p.state_numel = int(self._lib.dsoft_plan_state_bytes(h)) // 4
            p.scratch_numel = int(self._lib.dsoft_plan_scratch_bytes(h)) // 4
            p.fwd_scratch_numel = int(self._lib.dsoft_plan_forward_scratch_bytes(h)) // 4
            p.flops = float(self._lib.dsoft_plan_algorithmic_flops(h))
            p.launches_fwd = int(self._lib.dsoft_plan_launches_forward(h))
            p.launches_bwd = int(self._lib.dsoft_plan_launches_backward(h))
            p.dino_col = int(self._lib.dsoft_plan_dino_col_offset(h))
            info = (C.c_longlong * 12)()
            _cabi.check(self._lib.dsoft_plan_symw_info(h, info, 12), "dsoft_plan_symw_info")
            p.symw = _SymW(list(info), shape.world, shape.rank) if info[0] else None
            # weighted CE at world > 1: the row-std block in `state` (offset, floats per rank, directions) that the
            # forward all-gathers between phases 5 and 6, and the widened per-row statistics of lse_local
            ws = (C.c_longlong * 3)()
            _cabi.check(self._lib.dsoft_plan_wsigma_info(h, ws, 3), "dsoft_plan_wsigma_info")
            p.wsig = (int(ws[0]), int(ws[1]), int(ws[2])) if ws[1] else None
            p.lse_rows = int(self._lib.dsoft_plan_lse_rows(h))
            p.shape = shape
            self._plans[key] = p
        return p

    @staticmethod
    def _stream(t: torch.Tensor):
        # the C side works on the CUDA runtime's current device: make it the tensors' device (a process that
        # holds several GPUs may call the loss for a tensor that does not live on the current one)
        if torch.cuda.current_device() != t.device.index:
            torch.cuda.set_device(t.device)
        return torch.cuda.current_stream(t.device).cuda_stream

    def pack(self, plan, image, text, student, dino, gathered):
        image, text = _rowmajor(image), _rowmajor(text)
        student = None if student is None else _rowmajor(student)
        dino = None if dino is None else _rowmajor(dino)
        d = lambda t: 0 if t is None else _DTYPES[t.dtype]
        ld = lambda t: 0 if t is None else t.stride(0)
        _cabi.check(
            self._lib.dsoft_pack(plan.handle, _ptr(image), d(image), ld(image), _ptr(text), d(text), ld(text),
                                 _ptr(student), d(student), ld(student), _ptr(dino), d(dino), ld(dino),
                                 _ptr(gathered), self._stream(gathered)),
            "dsoft_pack",
        )

    def head_forward(self, plan, gathered, w1, b1, w2, b2, hidden):
        """Projection head on the tile kernels: image columns of `gathered` -> student columns (+ hidden)."""
        _cabi.check(
            self._lib.dsoft_head_forward(plan.handle, _ptr(gathered), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2),
                                         0 if hidden is None else hidden.shape[1], _ptr(hidden),
                                         self._stream(gathered)),
            "dsoft_head_forward",
        )

    def concurrency(self, plan) -> int:
        """0: the C side launches serially, 1: on forked lanes, 2: serially because the kernel recorder is on."""
        return int(self._lib.dsoft_plan_concurrency(plan.handle))

    @staticmethod
    def _lam(lambdas):
        import ctypes as C

        return (C.c_float * 4)(*[float(x) for x in lambdas])

    def forward(self, plan, gathered, logit_scale, lambdas, state, scratch, lse_local, losses, dbg=None, phase=0):
        """phase 0: whole forward; a plan with `symw`: 4 operand statistics, 1 soft part, 3 CLIP part, 2 finalize;
        a plan with `wsig`: 5 up to the weighted row stds, 6 the rest."""
        a = (plan.handle, _ptr(gathered), _ptr(logit_scale), self._lam(lambdas), _ptr(state), _ptr(scratch),
             _ptr(lse_local), _ptr(losses), _ptr(dbg), self._stream(gathered))
        if phase == 0:
            _cabi.check(self._lib.dsoft_forward(*a), "dsoft_forward")
        else:
            _cabi.check(self._lib.dsoft_forward_phase(*a, phase), "dsoft_forward_phase")

    def backward(self, plan, gathered, state, scratch, lse_all, gout, lambdas, d_image, d_text, d_student, d_scale,
                 phase=0):
        """phase 0: whole backward; a plan with `symw`: 4 relayout + fp16 operands, 1 soft part, 3 CLIP part, 2 finalize."""
        a = (plan.handle, _ptr(gathered), _ptr(state), _ptr(scratch), _ptr(lse_all), _ptr(gout), self._lam(lambdas),
             _ptr(d_image), _ptr(d_text), _ptr(d_student), _ptr(d_scale), self._stream(gathered))
        if phase == 0:
            _cabi.check(self._lib.dsoft_backward(*a), "dsoft_backward")
        else:
            _cabi.check(self._lib.dsoft_backward_phase(*a, phase), "dsoft_backward_phase")


_cuda_backend: Optional[CudaBackend] = None


def _default_backend(device: torch.device) -> CudaBackend:
    global _cuda_backend
    if device.type != "cuda":
        raise RuntimeError(
            "ClipLossWithDINOEnhancements (B200 build) needs CUDA tensors on an sm_100 device; "
            f"got device '{device}'. There is no CPU fallback."
        )
    if _cuda_backend is None:
        _cuda_backend = CudaBackend()
    return _cuda_backend


# ---- two-phase backward (DSOFT_F_GMAT, include/dsoft.h) ------------------------------------------------
# "auto": run the backward through fp16 logit-gradient matrices (2 B per element of up to four [b, B] blocks of
# backward scratch) whenever they fit in GMAT_FRACTION of the device memory that is free right now; otherwise
# use the fused backward, which never allocates anything of size b x B.  "always" / "never" force one path.
GMAT = os.environ.get("DSOFT_GMAT", "auto")
GMAT_FRACTION = 0.5


_gmat_decisions = {}


def _gmat_fits(b, W, soft, text, soft_local, dev) -> bool:
    if GMAT == "never":
        return False
    if GMAT == "always":
        return True
    if dev.type != "cuda":
        return False
    key = (b, W, soft, text, soft_local, dev.index)
    hit = _gmat_decisions.get(key)
    if hit is not None:  # decided when this shape was first seen: no driver query on the step path
        return hit
    _gmat_decisions[key] = _gmat_fits_now(b, W, soft, text, soft_local, dev)
    return _gmat_decisions[key]


def _gmat_fits_now(b, W, soft, text, soft_local, dev) -> bool:
    B = b * W
    cols_s = b if soft_local else B
    n_soft = (1 if soft else 0) + (1 if text else 0)
    if W == 1:  # one CLIP matrix, but a row-scaled second copy of each soft matrix (triangular backward)
        need = 2 * b * (B + 2 * n_soft * cols_s)
    else:
        need = 2 * b * (2 * B + n_soft * cols_s)
    free, _total = torch.cuda.mem_get_info(dev)
    cached = torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)
    return need <= GMAT_FRACTION * (free + cached)


class _FnConfig:
    __slots__ = ("backend", "world", "rank", "group", "flags", "teacher_temp", "text_temp", "lambdas", "rho",
                 "c_clip", "head_dp")


# ---- fused projection head (SURVEY 8f-3) ----------------------------------------------------------------
# Under bf16 autocast (how train.py:285 calls the loss) a plain Linear / Linear-ReLU-Linear head runs on the tile
# kernels (dsoft_head_forward): bf16 operands, fp32 accumulation, bias + ReLU + bf16 rounding in the epilogue -
# the arithmetic autocast gives nn.Linear - and its output lands in the student columns of the packed buffer, so
# there is no student tensor, no cast and no pack pass.  The backward of the head (five small GEMMs) stays on
# cuBLAS, issued directly from _DinoSoftFn.backward.
FUSED_HEAD: bool = True  # False: the PyTorch head (tests compare the two)


def _fusable_head(module, image: torch.Tensor):
    """(w1, b1, w2, b2) of a head dsoft_head_forward can run, else None."""
    if not FUSED_HEAD or module is None or image.device.type != "cuda":
        return None
    if not (torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == torch.bfloat16):
        return None  # fp32 callers get fp32 nn.Linear arithmetic
    if isinstance(module, nn.Linear):
        lin = [module]
    elif (isinstance(module, nn.Sequential) and len(module) == 3 and isinstance(module[0], nn.Linear)
          and isinstance(module[1], nn.ReLU) and isinstance(module[2], nn.Linear)):
        lin = [module[0], module[2]]
    else:
        return None  # LayerNorm / residual variants: PyTorch
    for m in lin:
        if m.bias is None or m.weight.device != image.device or m.in_features % 8 or m.out_features % 8:
            return None
    if len(lin) == 1:
        return lin[0].weight, lin[0].bias, None, None
    return lin[0].weight, lin[0].bias, lin[1].weight, lin[1].bias


class _DinoSoftFn(torch.autograd.Function):
    """(image, text, logit_scale, student_raw, dino) ->
    [classic_loss, soft_imgimg, soft_texttext, soft_loss, total_loss, weighted_loss], dbg  (loss composition
    loss.py:397, 466, 473-477 is done by the finalize kernels: ~12 tiny PyTorch kernels fewer per step; dbg is the
    non-differentiable diagnostics array of the weighted branch, or an empty tensor)."""

    @staticmethod
    def forward(ctx, image, text, logit_scale, student, dino, cfg: _FnConfig, w1=None, b1=None, w2=None, b2=None):
        be = cfg.backend
        dev = image.device
        b, D = image.shape
        W, r = cfg.world, cfg.rank
        soft = bool(cfg.flags & _cabi.DSOFT_F_SOFT)
        weighted = bool(cfg.flags & _cabi.DSOFT_F_WEIGHTED)
        use_dino = soft or weighted
        needs_grad = any(ctx.needs_input_grad[:4]) or any(ctx.needs_input_grad[6:])
        fused_head = w1 is not None  # the head runs inside (dsoft_head_forward); `student` is None
        flags = cfg.flags
        # weighted plans take the two-phase backward unless GMAT == "never" (the memory rule does not cover their
        # matrices); when its scratch cannot be allocated, the backward below falls back to the fused form
        if needs_grad and ((weighted and GMAT != "never") or
                           _gmat_fits(b, W, soft, bool(flags & _cabi.DSOFT_F_TEXT),
                                      bool(flags & _cabi.DSOFT_F_SOFT_LOCAL), dev)):
            flags |= _cabi.DSOFT_F_GMAT
        shape = _cabi.Shape(
            b=b, world=W, rank=r, D=D,
            Dp=((cfg.head_dp if fused_head else student.shape[1]) if ((student is not None or fused_head) and soft)
                else 0),
            Dd=(dino.shape[1] if (dino is not None and use_dino) else 0),
            flags=flags, teacher_temp=cfg.teacher_temp, text_temp=cfg.text_temp, rho=cfg.rho, c_clip=cfg.c_clip,
        )
        plan = be.plan(shape, dev) if dev.type == "cuda" else be.plan(shape)
        gathered = torch.empty((b * W, plan.row_elems), dtype=torch.bfloat16, device=dev)
        lazy_dino = isinstance(dino, DinoRows)
        be.pack(plan, image.detach(), text.detach(), None if student is None or not soft else student.detach(),
                None if (dino is None or not use_dino or lazy_dino) else dino.detach(), gathered)
        hidden = w1b = w2b = None
        if fused_head:
            w1b = w1.detach().to(torch.bfloat16)
            w2b = None if w2 is None else w2.detach().to(torch.bfloat16)
            if w2 is not None:
                hidden = torch.empty((b, w1.shape[0]), dtype=torch.bfloat16, device=dev)
            be.head_forward(plan, gathered, w1b, b1.detach().float(), w2b,
                            None if b2 is None else b2.detach().float(), hidden)
        if lazy_dino and use_dino:
            # device feature store: the rows are gathered by index straight into the DINO columns of the packed
            # buffer (range check on the device), replacing train.py:250-280's CPU gather + H2D copy
            dino.store.gather_into_packed(dino, gathered, r * b, plan.dino_col)
        if W > 1:
            # the only feature exchange of the path: one all-gather of the packed bf16 rows (loss.py:23-81)
            dist.all_gather_into_tensor(gathered.view(-1), gathered[r * b:(r + 1) * b].view(-1), group=cfg.group)
        state = torch.empty(plan.state_numel, dtype=torch.float32, device=dev)
        scratch = torch.empty(plan.fwd_scratch_numel, dtype=torch.float32, device=dev)
        lse_all = torch.empty((W, getattr(plan, "lse_rows", 5), b), dtype=torch.float32, device=dev)
        losses = torch.empty(6, dtype=torch.float32, device=dev)
        dbg = torch.empty(_cabi.DBG_N if weighted else 0, dtype=torch.float32, device=dev)
        ls = logit_scale.detach().to(device=dev, dtype=torch.float32).reshape(1).contiguous()
        if getattr(plan, "symw", None) is not None:
            # symmetric soft tiles across ranks: the column sums this rank computed for other ranks' rows travel
            # (6 floats per row and owner) while the CLIP tile kernels run; the finalize kernel needs both
            fargs = (plan, gathered, ls, cfg.lambdas, state, scratch, lse_all[r], losses, None)
            plan.symw.run(dev, be.concurrency(plan), lambda ph: be.forward(*fargs, phase=ph),
                          lambda: plan.symw.exchange_forward(scratch, cfg.group))
        elif getattr(plan, "wsig", None) is not None:
            # weighted CE at world > 1: beta is the median of the row stds of all B rows, so the forward pauses once
            # for their all-gather (ndir floats per sample), in place in `state`
            fargs = (plan, gathered, ls, cfg.lambdas, state, scratch, lse_all[r], losses, dbg)
            be.forward(*fargs, phase=5)
            off, n, _ = plan.wsig
            sig = state[off:off + W * n]
            dist.all_gather_into_tensor(sig, sig[r * n:(r + 1) * n], group=cfg.group)
            be.forward(*fargs, phase=6)
        else:
            be.forward(plan, gathered, ls, cfg.lambdas, state, scratch, lse_all[r], losses, dbg if weighted else None)
        if W > 1 and needs_grad:
            # column-side soft-max statistics of the other ranks' rows (5 floats per sample; weighted CE: 3 more per
            # modulated direction)
            dist.all_gather_into_tensor(lse_all.view(-1), lse_all[r].view(-1), group=cfg.group)
        ctx.save_for_backward(gathered, state, lse_all, hidden, w1b, w2b)
        ctx.plan, ctx.cfg = plan, cfg
        ctx.fused_head = fused_head
        ctx.meta = (image.dtype, text.dtype, logit_scale.dtype, logit_scale.shape,
                    None if student is None else student.dtype, b, D, shape.Dp)
        ctx.mark_non_differentiable(dbg)
        return losses, dbg

    @staticmethod
    @once_differentiable
    def backward(ctx, gout, _gdbg=None):
        gathered, state, lse_all, hidden, w1b, w2b = ctx.saved_tensors
        plan, be = ctx.plan, ctx.cfg.backend
        idt, tdt, sdt, sshape, zdt, b, D, Dp = ctx.meta
        dev = gathered.device
        gout = gout.to(torch.float32).contiguous()
        d_image = torch.empty((b, D), dtype=torch.float32, device=dev)
        d_text = torch.empty((b, D), dtype=torch.float32, device=dev)
        d_student = torch.empty((b, Dp), dtype=torch.float32, device=dev) if Dp > 0 else None
        d_scale = torch.empty(1, dtype=torch.float32, device=dev)
        try:
            scratch = torch.empty(plan.scratch_numel, dtype=torch.float32, device=dev)
        except torch.cuda.OutOfMemoryError:
            # the fp16 logit-gradient matrices fitted when this shape was first seen but do not now: the saved
            # forward state does not depend on the backward implementation, so run the fused backward instead
            s = plan.shape
            if not (s.flags & _cabi.DSOFT_F_GMAT):
                raise
            for key in [k for k in _gmat_decisions if k[0] == s.b and k[1] == s.world]:
                _gmat_decisions[key] = False
            plan = be.plan(_cabi.Shape(b=s.b, world=s.world, rank=s.rank, D=s.D, Dp=s.Dp, Dd=s.Dd,
                                       flags=s.flags & ~_cabi.DSOFT_F_GMAT, teacher_temp=s.teacher_temp,
                                       text_temp=s.text_temp, rho=s.rho, c_clip=s.c_clip), dev)
            scratch = torch.empty(plan.scratch_numel, dtype=torch.float32, device=dev)
        args = (plan, gathered, state, scratch, lse_all, gout, ctx.cfg.lambdas, d_image, d_text, d_student, d_scale)
        if getattr(plan, "symw", None) is not None:
            # ... and the transposed gradient products (the reduce-scatter of `_AllGather.backward`, loss.py:59-64,
            # restricted to the soft terms and to the half of the blocks the other rank did not compute itself),
            # next to the CLIP logit-gradient kernels and gradient GEMMs
            plan.symw.run(dev, be.concurrency(plan), lambda ph: be.backward(*args, phase=ph),
                          lambda: plan.symw.exchange_backward(scratch, ctx.cfg.group))
        else:
            be.backward(*args)
        g_student = None
        if zdt is not None:
            g_student = d_student.to(zdt) if d_student is not None else None
        g_head = (None, None, None, None)
        if ctx.fused_head:
            # head backward in the arithmetic autocast gives the reference (bf16 operands, fp32 accumulation), on
            # cuBLAS: dZ -> (dW2, db2, dH) -> ReLU mask -> (dW1, db1, dX); dX joins d_image.  The parameter
            # gradients keep the fp32 accumulator (autocast would round them to bf16, up to 2^-8 relative)
            s = plan.shape
            r0 = s.rank * b
            x = gathered[r0:r0 + b, :D]  # image columns of this rank's rows (strided view)
            dz = d_student.to(torch.bfloat16)
            f32 = torch.float32
            if w2b is None:
                g_head = (torch.mm(dz.t(), x, out_dtype=f32), d_student.sum(0), None, None)
                d_image += (dz @ w1b).float()
            else:
                dh = torch.ops.aten.threshold_backward(dz @ w2b, hidden, 0.0)
                g_head = (torch.mm(dh.t(), x, out_dtype=f32), dh.sum(0, dtype=f32),
                          torch.mm(dz.t(), hidden, out_dtype=f32), d_student.sum(0))
                d_image += (dh @ w1b).float()
        return (d_image.to(idt), d_text.to(tdt), d_scale.reshape(sshape).to(sdt), g_student, None, None) + g_head


# --------------------------------------------------------------------------------------------------
# denominator-modulated ("weighted") CE branch, loss.py:416-471 + diagnostics loss.py:479-595
# --------------------------------------------------------------------------------------------------
# Runs inside libdsoft.so (DSOFT_F_WEIGHTED): three tile passes per direction over the CLIP and DINO Gram tiles
# (row statistics c_a = sum_j p r and the row std of the logits -> device-side median -> beta; log-sum-exp of the
# shifted logits; diagnostics) and one logit-gradient pass in the backward.  Nothing of size B x B is stored and beta
# never visits the host (the reference calls `.item()` twice per step).  At world_size > 1 (`weighted_scope="global"`)
# every rank runs its row block of the global problem: one extra all-gather of the row stds in the forward, and the
# per-row statistics the backward's column side needs travel with the existing LSE all-gather.  The loss terms and
# diagnostics are per rank (means over the rank's rows); beta_img / beta_txt are the global values.
DBG_KEYS = (  # index into the dbg array of dsoft_forward (include/dsoft.h)
    ("pc_err_img", 0), ("pc_err_txt", 1), ("diag_max_img", 2), ("diag_max_txt", 3),
    ("delta_img_max", 4), ("delta_img_mean", 5), ("delta_img_std", 6),
    ("delta_txt_max", 7), ("delta_txt_mean", 8), ("delta_txt_std", 9),
    ("l1_prob_shift_img", 10), ("l1_prob_shift_txt", 11),
    ("corr_rhat_dprob_img", 12), ("corr_rhat_dprob_txt", 13),
    ("ce_img_base", 14), ("ce_txt_base", 15), ("ce_img_mod", 16), ("ce_txt_mod", 17),
    ("pos_frac_img", 18), ("neg_frac_img", 19), ("pos_frac_txt", 20), ("neg_frac_txt", 21),
    ("beta_img", 22), ("beta_txt", 23),
)


def _normalize_out_dtype(x: torch.Tensor) -> torch.dtype:
    """dtype of F.normalize(x) where the reference computes it (inside train.py's autocast region or not)."""
    if x.dtype == torch.float32 or x.dtype == torch.float64:
        return x.dtype
    try:
        autocast = torch.is_autocast_enabled(x.device.type)
    except TypeError:  # older torch: no device argument
        autocast = torch.is_autocast_enabled()
    return torch.float32 if autocast else x.dtype


# --------------------------------------------------------------------------------------------------
# the loss module (same class name / ctor / forward signature as loss.py:190-300)
# --------------------------------------------------------------------------------------------------
class ClipLossWithDINOEnhancements(nn.Module):
    def __init__(
        self,
        local_loss: bool = False,
        gather_with_grad: bool = False,
        cache_labels: bool = False,
        rank: int = 0,
        world_size: int = 1,
        use_horovod: bool = False,
        soft_scope: str = "global",
        process_group=None,
        sync_projection: bool = True,
        weighted_scope: Optional[str] = None,
    ):
        super().__init__()
        self.local_loss = local_loss
        self.gather_with_grad = gather_with_grad
        self.cache_labels = cache_labels
        self.rank = rank
        self.world_size = world_size
        self.use_horovod = use_horovod
        if soft_scope not in ("global", "local"):
            raise ValueError(f"soft_scope must be 'global' or 'local', got {soft_scope!r}")
        self.soft_scope = soft_scope
        if weighted_scope not in (None, "global"):
            raise ValueError(f"weighted_scope must be None or 'global', got {weighted_scope!r}")
        # None: the reference's behaviour (the lambda_weighted branch fails at world_size > 1); "global": rank r
        # computes rows [r b, (r+1) b) of the branch on the concatenated batch (DESIGN.md section 1)
        self.weighted_scope = weighted_scope
        self.process_group = process_group
        self.sync_projection = sync_projection

        self.image_to_dino_proj = None

        self.prev_num_logits = 0
        self.labels = {}  # cache per-device
        self._backend = None  # resolved on first use; tests may inject a stand-in for host-logic checks

    # ------------------- Projection helper (loss.py:214-238) -------------------
    def init_proj(self, embed_dim, dino_dim, device, projection_type="mlp", residual=False, layernorm=False):
        if self.image_to_dino_proj is None:
            if projection_type == "linear":
                proj = nn.Linear(embed_dim, dino_dim)
            elif projection_type == "mlp":
                hidden_dim = (embed_dim + dino_dim) // 2
                layers = [nn.Linear(embed_dim, hidden_dim), nn.ReLU(), nn.Linear(hidden_dim, dino_dim)]
                if layernorm:
                    layers.append(nn.LayerNorm(dino_dim))
                proj = nn.Sequential(*layers)
            else:
                raise ValueError(f"Unknown projection_type: {projection_type}")
            self.image_to_dino_proj = proj.to(device)
            if self.world_size > 1 and self.sync_projection and self.soft_scope == "global":
                # the reference leaves every rank with its own random head (SURVEY.md section 3d); with
                # global soft targets the student columns must come from one head, so rank 0's is used
                for p in self.image_to_dino_proj.parameters():
                    dist.broadcast(p.data, src=0, group=self.process_group)

    # --------------------------- helpers (loss.py:241-274) -------------------------------------
    def get_ground_truth(self, device: torch.device, num_logits: int) -> torch.Tensor:
        dev_key = str(device)
        if self.prev_num_logits != num_logits or dev_key not in self.labels:
            labels = torch.arange(num_logits, device=device, dtype=torch.long)
            if self.world_size > 1 and self.local_loss:
                labels += num_logits * self.rank
            if self.cache_labels:
                self.labels[dev_key] = labels
            self.prev_num_logits = num_logits
        else:
            labels = self.labels[dev_key]
        return labels

    def get_logits(self, image_features: torch.Tensor, text_features: torch.Tensor, logit_scale: torch.Tensor):
        """API parity with loss.py:254-274 (materialises the logits; NOT used by ``forward``)."""
        if self.world_size > 1:
            all_image_features, all_text_features = gather_features(
                image_features, text_features, local_loss=self.local_loss,
                gather_with_grad=self.gather_with_grad, rank=self.rank, world_size=self.world_size,
                use_horovod=self.use_horovod,
            )
            if self.local_loss:
                logits_per_image = logit_scale * (image_features @ all_text_features.T)
                logits_per_text = logit_scale * (text_features @ all_image_features.T)
            else:
                logits_per_image = logit_scale * (all_image_features @ all_text_features.T)
                logits_per_text = logits_per_image.T
        else:
            logits_per_image = logit_scale * (image_features @ text_features.T)
            logits_per_text = logit_scale * (text_features @ image_features.T)
        return logits_per_image, logits_per_text

    # ------------------------------ forward (loss.py:292-607) ----------------------------------
    def forward(
        self,
        image_features: torch.Tensor,
        text_features: torch.Tensor,
        logit_scale: torch.Tensor,
        dino_features: Optional[torch.Tensor] = None,
        args=None,
        output_dict: bool = False,
    ):
        device = image_features.device
        B = image_features.shape[0]
        g = getattr

        use_projection = g(args, "use_projection", True)
        projection_type = g(args, "projection_type", "mlp")
        use_layernorm = g(args, "use_layernorm", False)
        residual_projection = g(args, "residual_projection", False)
        residual_alpha = g(args, "residual_alpha", None)

        if self.use_horovod:
            raise NotImplementedError("Horovod is not supported by the B200 DINO-Soft path (NCCL only)")
        if self.world_size > 1 and not self.local_loss:
            # the reference builds [WB, WB] logits against labels of the local batch and cross_entropy
            # raises (loss.py:269, 314-318); keep the failure instead of inventing semantics
            raise ValueError(
                f"Expected input batch_size ({B * self.world_size}) to match target batch_size ({B})."
            )
        lambda_weighted = float(g(args, "lambda_weighted", 0.0))
        weighted_on = lambda_weighted > 0.0 and dino_features is not None and B > 1  # loss.py:422
        if weighted_on and self.world_size > 1 and self.weighted_scope is None:
            # the reference builds r and the diagonal mask from the LOCAL batch against [b, B] logits
            # (loss.py:423-446) and fails in the first broadcast; keep the failure
            raise RuntimeError(
                f"The size of tensor a ({B * self.world_size}) must match the size of tensor b ({B}) at "
                "non-singleton dimension 1 (the lambda_weighted branch is single-rank only, loss.py:416-471)"
            )

        lambda_soft = float(g(args, "lambda_soft", 0.0))
        soft_mode = g(args, "soft_mode", "none")
        soft_on = lambda_soft > 0.0 and soft_mode == "kl_teacher" and dino_features is not None
        text_on = soft_on and bool(g(args, "soft_dino_to_text", False)) and float(g(args, "text_lambda", 0.2)) > 0.0

        # ----- projection head (loss.py:322-347); stays in PyTorch/cuBLAS, its output is the student operand
        student = None
        head = None
        if dino_features is not None and use_projection:
            self.init_proj(
                embed_dim=image_features.size(-1), dino_dim=dino_features.size(-1), device=device,
                projection_type=projection_type, layernorm=use_layernorm,
            )
            if soft_on and not residual_projection and self._backend is None:
                head = _fusable_head(self.image_to_dino_proj, image_features)
            if soft_on and head is None:
                raw_proj = self.image_to_dino_proj(image_features)
                student = raw_proj
                if residual_projection and raw_proj.shape == image_features.shape:
                    if residual_alpha is None:
                        student = image_features + raw_proj
                    else:
                        student = residual_alpha * image_features + (1 - residual_alpha) * raw_proj

        flags = 0
        teacher_temp = text_temp = 0.0
        if soft_on:
            flags |= _cabi.DSOFT_F_SOFT
            # tau_t / tau_txt are materialised in the dtype of Zs / Tn = F.normalize(...) by the reference
            # (loss.py:368-369, 392-393); under CUDA autocast F.normalize returns fp32 whatever its input is
            # (`norm` is on autocast's fp32 list), so the temperatures are rounded through THAT dtype
            zs_dtype = _normalize_out_dtype(student if student is not None else image_features)
            teacher_temp = float(torch.as_tensor(float(g(args, "teacher_temp", 0.15)), dtype=zs_dtype))
            if text_on:
                flags |= _cabi.DSOFT_F_TEXT
                text_temp = float(
                    torch.as_tensor(float(g(args, "text_student_temp", 0.05)),
                                    dtype=_normalize_out_dtype(text_features))
                )
            if self.world_size > 1 and self.soft_scope == "local":
                flags |= _cabi.DSOFT_F_SOFT_LOCAL
        if self.world_size > 1 and not self.gather_with_grad:
            flags |= _cabi.DSOFT_F_ROW_ONLY
        if weighted_on:
            flags |= _cabi.DSOFT_F_WEIGHTED
            if bool(g(args, "weight_text_symmetry", False)):
                flags |= _cabi.DSOFT_F_WSYM

        lambda_original = float(g(args, "lambda_original", 1.0))
        text_lambda = float(g(args, "text_lambda", 0.2)) if text_on else 0.0
        cfg = _FnConfig()
        cfg.backend = self._backend if self._backend is not None else _default_backend(device)
        cfg.world, cfg.rank, cfg.group = self.world_size, self.rank, self.process_group
        cfg.flags, cfg.teacher_temp, cfg.text_temp = flags, teacher_temp, text_temp
        cfg.lambdas = (lambda_original, lambda_soft if soft_on else 0.0, text_lambda,
                       lambda_weighted if weighted_on else 0.0)
        cfg.rho, cfg.c_clip = float(g(args, "rho", 0.1)), float(g(args, "c_clip", 1.0))
        cfg.head_dp = 0
        head_args = (None, None, None, None)
        if student is None and dino_features is not None and use_projection and soft_on and head is not None:
            cfg.head_dp = (head[2] if head[2] is not None else head[0]).shape[0]
            head_args = head

        terms, dbg_arr = _DinoSoftFn.apply(
            image_features, text_features, logit_scale, student,
            dino_features if (soft_on or weighted_on) else None, cfg, *head_args
        )
        classic_loss = terms[0]
        soft_loss = terms[3] if soft_on else torch.zeros((), device=device)
        weighted_loss = terms[5] if weighted_on else torch.zeros((), device=device, dtype=classic_loss.dtype)
        total_loss = terms[4]  # loss.py:473-477, composed on the device
        dbg = {}
        if weighted_on:
            # 0-dim views of the device array: formatting one (train.py:360-364, every 300 steps) is what syncs
            dbg = {k: dbg_arr[i] for k, i in DBG_KEYS}
            dbg["rho"], dbg["clip_c"] = cfg.rho, cfg.c_clip
        if output_dict:
            return {
                "total_loss": total_loss,
                "classic_loss": classic_loss,
                "soft_loss": soft_loss,
                "weighted_loss": weighted_loss,
                "dbg": dbg,
            }
        # the reference returns None when output_dict is False (loss.py:598-607) - preserved


def install_into_open_clip(open_clip_module=None, siglip=False, distill=False):
    """Make the reference's ``create_loss`` (factory.py:566-576) build this class.

    ``open_clip.factory`` imports the class by name at import time (factory.py:25-34), so both module
    attributes are patched; ``train.py`` needs no change.  ``siglip=True`` also patches every binding of
    ``SigLipLoss`` (the ``--siglip`` objective) with ``siglip.SigLipLoss``; off by default, so that existing callers
    keep upstream's SigLIP loss.  ``distill=True`` likewise patches ``DistillClipLoss`` (the ``--distill`` objective)
    with ``distill.DistillClipLoss``; off by default."""
    import importlib

    loss_mod = importlib.import_module("open_clip.loss") if open_clip_module is None else open_clip_module.loss
    factory_mod = importlib.import_module("open_clip.factory") if open_clip_module is None else open_clip_module.factory
    if not hasattr(loss_mod, "_reference_ClipLossWithDINOEnhancements"):
        loss_mod._reference_ClipLossWithDINOEnhancements = loss_mod.ClipLossWithDINOEnhancements
    loss_mod.ClipLossWithDINOEnhancements = ClipLossWithDINOEnhancements
    factory_mod.ClipLossWithDINOEnhancements = ClipLossWithDINOEnhancements
    if hasattr(loss_mod, "CyCLIPLoss"):  # the CyCLIP drop-in (factory.py:537-549; train.py:316 isinstance check)
        from .cyclip import CyCLIPLoss

        if not hasattr(loss_mod, "_reference_CyCLIPLoss"):
            loss_mod._reference_CyCLIPLoss = loss_mod.CyCLIPLoss
        loss_mod.CyCLIPLoss = CyCLIPLoss
        factory_mod.CyCLIPLoss = CyCLIPLoss
        import sys

        train_mod = sys.modules.get("open_clip_train.train")  # train.py:16 binds the name at import, :316 isinstance
        if train_mod is not None and hasattr(train_mod, "CyCLIPLoss"):
            train_mod.CyCLIPLoss = CyCLIPLoss
    if siglip and hasattr(loss_mod, "SigLipLoss"):
        from .siglip import SigLipLoss
        import sys

        if not hasattr(loss_mod, "_reference_SigLipLoss"):
            loss_mod._reference_SigLipLoss = loss_mod.SigLipLoss
        loss_mod.SigLipLoss = SigLipLoss
        factory_mod.SigLipLoss = SigLipLoss
        train_mod = sys.modules.get("open_clip_train.train")
        if train_mod is not None and hasattr(train_mod, "SigLipLoss"):
            train_mod.SigLipLoss = SigLipLoss
    if distill and hasattr(loss_mod, "DistillClipLoss"):
        from .distill import DistillClipLoss
        import sys

        if not hasattr(loss_mod, "_reference_DistillClipLoss"):
            loss_mod._reference_DistillClipLoss = loss_mod.DistillClipLoss
        loss_mod.DistillClipLoss = DistillClipLoss
        factory_mod.DistillClipLoss = DistillClipLoss
        train_mod = sys.modules.get("open_clip_train.train")
        if train_mod is not None and hasattr(train_mod, "DistillClipLoss"):
            train_mod.DistillClipLoss = DistillClipLoss
    return ClipLossWithDINOEnhancements


def uninstall_from_open_clip(open_clip_module=None):
    """Undo ``install_into_open_clip`` (A/B runs of the reference's loss and this one in one process)."""
    import importlib

    loss_mod = importlib.import_module("open_clip.loss") if open_clip_module is None else open_clip_module.loss
    factory_mod = importlib.import_module("open_clip.factory") if open_clip_module is None else open_clip_module.factory
    ref = getattr(loss_mod, "_reference_ClipLossWithDINOEnhancements", None)
    if ref is not None:
        loss_mod.ClipLossWithDINOEnhancements = ref
        factory_mod.ClipLossWithDINOEnhancements = ref
    cyc = getattr(loss_mod, "_reference_CyCLIPLoss", None)
    if cyc is not None:
        loss_mod.CyCLIPLoss = cyc
        factory_mod.CyCLIPLoss = cyc
        import sys

        train_mod = sys.modules.get("open_clip_train.train")
        if train_mod is not None and hasattr(train_mod, "CyCLIPLoss"):
            train_mod.CyCLIPLoss = cyc
    sig = getattr(loss_mod, "_reference_SigLipLoss", None)
    if sig is not None:
        import sys

        loss_mod.SigLipLoss = sig
        factory_mod.SigLipLoss = sig
        train_mod = sys.modules.get("open_clip_train.train")
        if train_mod is not None and hasattr(train_mod, "SigLipLoss"):
            train_mod.SigLipLoss = sig
    dcl = getattr(loss_mod, "_reference_DistillClipLoss", None)
    if dcl is not None:
        import sys

        loss_mod.DistillClipLoss = dcl
        factory_mod.DistillClipLoss = dcl
        train_mod = sys.modules.get("open_clip_train.train")
        if train_mod is not None and hasattr(train_mod, "DistillClipLoss"):
            train_mod.DistillClipLoss = dcl
    return ref
