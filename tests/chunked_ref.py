"""Row-blocked fp64 evaluation of the DINO-Soft loss (world size 1) for batch sizes where the B x B matrices do
not fit: TEST INFRASTRUCTURE (a checker next to oracle/dinosoft_oracle.py, which it is validated against on the
CPU by tests/test_chunked_ref.py).

Semantics restated (reference src/open_clip/loss.py): CLIP CE 313-319, projection + normalise 322-347, KL-teacher
term 356-384, text-text term 387-397, total 473-477.  Everything runs in fp64 on the device of the inputs.

  pass 1  row slabs of the four B x B matrices -> row / column log-sum-exps, the loss terms
  pass 2  d(logit_scale), which needs the finished column log-sum-exps
  blocks  for a sampled set of rows R: the exact gradient of the TOTAL loss w.r.t. image_R, text_R and the raw
          student rows, from  F = A + C  under autograd, where
            A = the loss rows R with their row operand live and every column operand constant, and
            C = sum_ji G[j, i] * logit[j, i](x_i)  over ALL rows j and the columns i in R, with
                G = d loss / d logit evaluated in fp64 without gradient
          (a logit depends on its row operand and on its column operand; A carries the first dependence and C
          the second, diagonal entries appear in both, as they must).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F


def _norm(x):
    return x / x.pow(2).sum(-1, keepdim=True).sqrt().clamp_min(1e-12)


class _RoundBF16STE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return g


def _head(x, hp):
    if hp is None:
        return None
    h = torch.relu(x @ hp["w0"].T + hp["b0"])
    return h @ hp["w1"].T + hp["b1"]


def _student_tau(scale: float) -> float:  # loss.py:166-175
    import math

    m = scale if scale > 10 else math.exp(scale)
    m = min(m, 100.0)
    return min(max(1.0 / m, 0.008), 0.02)


def chunked_reference(img, txt, dino, scale, head=None, blocks=(), lambdas=(1.0, 0.5, 0.5), teacher_temp=0.15,
                      text_temp=0.02, slab=2048, student_values=None):
    """img/txt [B, D], dino [B, Dd] (any float dtype, one device); head = dict(w0, b0, w1, b1) or None;
    blocks = iterable of (row0, nrows).  Returns loss terms (python floats), d_logit_scale and per block
    d_image / d_text / d_student (fp64 tensors).  student_values [B, Dp]: the (bf16-rounded) student operand the
    implementation under test really used; replaces the VALUE of the head output (gradients still flow through
    the head), see oracle.loss_and_grads.  With student_values and no head the student is a leaf: d_image and
    d_text are the loss side alone and d_student is the gradient the head's backward starts from."""
    dt = torch.float64
    dev = img.device
    lam_o, lam_s, lam_x = (float(v) for v in lambdas)
    s = float(scale)
    I, T = img.to(dt), txt.to(dt)
    hp = None if head is None else {k: v.to(device=dev, dtype=dt) for k, v in head.items()}
    B = I.shape[0]
    with torch.no_grad():
        raw = I if hp is None else torch.cat([_head(I[i:i + slab], hp) for i in range(0, B, slab)])
        S = raw.to(torch.bfloat16).to(dt) if hp is not None else raw
        if student_values is not None:
            S = student_values.to(dt)
        Z = _norm(_norm(S))
        Dn = _norm(dino.to(dt))
        Tn = _norm(T)
        tau_s, tau_t, tau_x = _student_tau(s), float(teacher_temp), float(text_temp)
        lse_it = torch.empty(B, dtype=dt, device=dev)
        lse_ti = torch.full((B,), -float("inf"), dtype=dt, device=dev)
        lt, ls, lx = (torch.empty(B, dtype=dt, device=dev) for _ in range(3))
        diag = (I * T).sum(-1)
        kl_s = torch.zeros((), dtype=dt, device=dev)
        kl_x = torch.zeros((), dtype=dt, device=dev)
        for r0 in range(0, B, slab):
            r1 = min(r0 + slab, B)
            idx = torch.arange(r0, r1, device=dev)
            L = s * (I[r0:r1] @ T.T)
            lse_it[r0:r1] = torch.logsumexp(L, dim=1)
            lse_ti = torch.logaddexp(lse_ti, torch.logsumexp(L, dim=0))
            St = (Dn[r0:r1] @ Dn.T) / tau_t
            St[idx - r0, idx] = -float("inf")  # loss.py:376-377
            lt[r0:r1] = torch.logsumexp(St, dim=1)
            logq = St - lt[r0:r1, None]
            q = logq.exp()
            Ss = (Z[r0:r1] @ Z.T) / tau_s
            ls[r0:r1] = torch.logsumexp(Ss, dim=1)
            logq[idx - r0, idx] = 0.0  # q = 0 there: xlogy(0, 0) = 0
            kl_s += (q * (logq - (Ss - ls[r0:r1, None]))).sum()
            Sx = (Tn[r0:r1] @ Tn.T) / tau_x
            lx[r0:r1] = torch.logsumexp(Sx, dim=1)
            kl_x += (q * (logq - (Sx - lx[r0:r1, None]))).sum()
        classic = 0.5 * ((lse_it - s * diag).mean() + (lse_ti - s * diag).mean())
        soft_img, soft_txt = kl_s / B, kl_x / B
        soft = soft_img + lam_x * soft_txt
        total = lam_o * classic + lam_s * soft
        # ---- pass 2: d total / d logit_scale = lam_o / (2B) * sum_ij (p_it[i,j] + p_ti[j,i] - 2 delta_ij) dot_ij
        dsc = torch.zeros((), dtype=dt, device=dev)
        for r0 in range(0, B, slab):
            r1 = min(r0 + slab, B)
            dot = I[r0:r1] @ T.T
            L = s * dot
            dsc += (((L - lse_it[r0:r1, None]).exp() + (L - lse_ti[None, :]).exp()) * dot).sum()
        dsc = lam_o * (dsc - 2.0 * diag.sum()) / (2.0 * B)
    out = dict(classic_loss=float(classic), soft_img=float(soft_img), soft_txt=float(soft_txt),
               soft_loss=float(soft), total_loss=float(total), d_logit_scale=float(dsc), blocks=[])

    for (b0, nb) in blocks:
        R = slice(b0, b0 + nb)
        ridx = torch.arange(b0, b0 + nb, device=dev)
        loc = torch.arange(nb, device=dev)
        im = I[R].clone().requires_grad_(True)
        tx = T[R].clone().requires_grad_(True)
        if hp is not None:
            st = _RoundBF16STE.apply(_head(im, hp))
            if student_values is not None:
                st = st + (student_values[R].to(dt) - st).detach()
            st.retain_grad()
        elif student_values is not None:  # the student as a leaf of its own: d_image is the loss side alone
            st = student_values[R].to(dt).clone().requires_grad_(True)
        else:
            st = im
        z = _norm(_norm(st))
        tn = _norm(tx)
        # ---- A: rows R, row operand live, columns constant
        Lr = s * (im @ T.T)
        Lr2 = s * (tx @ I.T)
        a_classic = ((torch.logsumexp(Lr, 1) - Lr[loc, ridx]).sum() + (torch.logsumexp(Lr2, 1) - Lr2[loc, ridx]).sum())
        with torch.no_grad():
            St = (Dn[R] @ Dn.T) / tau_t
            St[loc, ridx] = -float("inf")
            q = torch.softmax(St, dim=1)
        Ss = (z @ Z.T) / tau_s
        a_s = -(q * (Ss - torch.logsumexp(Ss, 1, keepdim=True))).sum()  # + const (sum q log q)
        Sx = (tn @ Tn.T) / tau_x
        a_x = -(q * (Sx - torch.logsumexp(Sx, 1, keepdim=True))).sum()
        A = lam_o * a_classic / (2.0 * B) + lam_s * (a_s + lam_x * a_x) / B
        # ---- C: columns R live, G = d loss / d logit for all rows j constant
        with torch.no_grad():
            onehot = torch.zeros(B, nb, dtype=dt, device=dev)
            onehot[ridx, loc] = 1.0
            G_it = ((s * (I @ T[R].T) - lse_it[:, None]).exp() - onehot) * (lam_o / (2.0 * B))   # [B, nb]
            G_ti = ((s * (T @ I[R].T) - lse_ti[:, None]).exp() - onehot) * (lam_o / (2.0 * B))
            Qc = (Dn @ Dn[R].T) / tau_t
            Qc[ridx, loc] = -float("inf")
            Qc = (Qc - lt[:, None]).exp()
            G_s = (((Z @ Z[R].T) / tau_s - ls[:, None]).exp() - Qc) * (lam_s / B)
            G_x = (((Tn @ Tn[R].T) / tau_x - lx[:, None]).exp() - Qc) * (lam_s * lam_x / B)
            M_it, M_ti = G_it.T @ I, G_ti.T @ T       # [nb, D]
            M_s, M_x = G_s.T @ Z, G_x.T @ Tn
        Cc = s * ((tx * M_it).sum() + (im * M_ti).sum()) + (z * M_s).sum() / tau_s + (tn * M_x).sum() / tau_x
        (A + Cc).backward()
        out["blocks"].append(dict(row0=b0, rows=nb, d_image=im.grad.detach(), d_text=tx.grad.detach(),
                                  d_student=None if st is im else st.grad.detach()))
    return out


def chunked_weighted_loss(img, txt, dino, scale, rho, c_clip, sym, slab=2048):
    """Row-blocked fp64 evaluation of the denominator-modulated CE (loss.py:416-471), forward only:
    0.5 * (CE(L_it + Delta_it) + CE(L_ti [+ Delta_ti]))."""
    dt = torch.float64
    dev = img.device
    I, T = img.to(dt), txt.to(dt)
    Dn = _norm(dino.to(dt))
    s = float(scale)
    B = I.shape[0]
    diag = s * (I * T).sum(-1)

    def one_direction(R, C, modulate):
        lse = torch.empty(B, dtype=dt, device=dev)
        cst = torch.empty(B, dtype=dt, device=dev)
        std = torch.empty(B, dtype=dt, device=dev)
        for r0 in range(0, B, slab):
            r1 = min(r0 + slab, B)
            idx = torch.arange(r0, r1, device=dev)
            L = s * (R[r0:r1] @ C.T)
            lse[r0:r1] = torch.logsumexp(L, dim=1)
            if modulate:
                r = 1.0 - (Dn[r0:r1] @ Dn.T).clamp(-1, 1)
                r[idx - r0, idx] = 0.0
                cst[r0:r1] = (torch.softmax(L, dim=1) * r).sum(1)
                std[r0:r1] = L.std(dim=1)
        if not modulate:
            return (lse - diag).mean()
        beta = rho * torch.median(std).clamp(min=1e-6) / c_clip
        ce = torch.zeros((), dtype=dt, device=dev)
        for r0 in range(0, B, slab):
            r1 = min(r0 + slab, B)
            idx = torch.arange(r0, r1, device=dev)
            L = s * (R[r0:r1] @ C.T)
            r = 1.0 - (Dn[r0:r1] @ Dn.T).clamp(-1, 1)
            r[idx - r0, idx] = 0.0
            delta = beta * (r - cst[r0:r1, None]).clamp(-c_clip, c_clip)
            delta[idx - r0, idx] = 0.0
            ce += (torch.logsumexp(L + delta, dim=1) - diag[r0:r1]).sum()
        return ce / B

    with torch.no_grad():
        return float(0.5 * (one_direction(I, T, True) + one_direction(T, I, bool(sym))))
