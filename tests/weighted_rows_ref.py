"""TEST INFRASTRUCTURE: fp64 restatement of the weighted CE branch at world size > 1 (`weighted_scope="global"`).

Rank r owns rows [r b, (r+1) b) of the branch on the concatenated batch of B = W b rows: beta comes from the row
stds of ALL B rows (one global value), the CE and the diagnostics are over the rank's row block only, with the
diagonal of local row i at column r b + i.  At one block (rows = all B) both functions reduce to the world-size-1
statements (`oracle.weighted_ce`, `weighted_ref.weighted_ce_branch`); tests/test_weighted_scope_host.py checks that.
"""
import torch
import torch.nn.functional as F

from weighted_ref import row_corr_mean


def _dissim_rows(dino, rows):
    """r = 1 - clamp(cos) of the DINO features with a zero diagonal, rows `rows` against all B columns."""
    with torch.no_grad():
        dn = F.normalize(dino, dim=-1)
        r = 1.0 - (dn[rows] @ dn.T).clamp(-1, 1)
        n = r.shape[0]
        r[torch.arange(n), torch.arange(rows.start, rows.start + n)] = 0.0
    return r


def _beta(full_logits, rho, c_clip):
    """rho * median(row std over all B rows) / c_clip; torch.median takes the lower middle value, no gradient."""
    with torch.no_grad():
        sigma = torch.median(full_logits.std(dim=1)).clamp(min=1e-6)
    return float(rho * sigma / c_clip)


def _shift(x, r, beta, c_clip, rows):
    """x + beta * clamp(r - E_p[r]) with p = soft-max of the unmodified rows (carries gradient), diagonal unshifted."""
    p = torch.softmax(x, dim=1)
    r_hat = (r - (p * r).sum(dim=1, keepdim=True)).clamp(min=-c_clip, max=c_clip)
    delta = (beta * r_hat).clone()
    n = x.shape[0]
    delta[torch.arange(n), torch.arange(rows.start, rows.start + n)] = 0.0
    return x + delta, delta, r_hat, p


def weighted_ce_global_rows(logits_it, logits_ti, dino, rows, rho, c_clip, text_sym):
    """One rank's weighted loss.  ``logits_it`` / ``logits_ti`` are the full [B, B] logits of the concatenated batch
    (image rows x text columns, text rows x image columns); only their rows ``rows`` reach the loss (the others only
    feed beta, without gradient), so a caller may pass the other rows detached.  Returns {loss, beta_img, beta_txt}."""
    B = dino.shape[0]
    if logits_it.shape != (B, B) or logits_ti.shape != (B, B):
        raise ValueError(f"need the full [{B}, {B}] logits of the concatenated batch")
    r = _dissim_rows(dino, rows)  # the DINO product is symmetric: the text direction uses the same rows
    labels = torch.arange(rows.start, rows.stop)
    beta_img = _beta(logits_it, rho, c_clip)
    it_tilde = _shift(logits_it[rows], r, beta_img, c_clip, rows)[0]
    beta_txt = 0.0
    if text_sym:
        beta_txt = _beta(logits_ti, rho, c_clip)
        ti_tilde = _shift(logits_ti[rows], r, beta_txt, c_clip, rows)[0]
    else:
        ti_tilde = logits_ti[rows]
    loss = 0.5 * (F.cross_entropy(it_tilde, labels) + F.cross_entropy(ti_tilde, labels))
    return {"loss": loss, "beta_img": beta_img, "beta_txt": beta_txt}


def weighted_ce_rows_branch(image_all, text_all, logit_scale, dino_all, rho, c_clip, text_sym, rows):
    """(weighted_loss, dbg) of one rank: the reference's diagnostic formulas (loss.py:479-595, as restated by
    weighted_ref.weighted_ce_branch) over the row block ``rows`` of the concatenated problem; beta_img / beta_txt are
    the global values, every other key is over the block's b x B entries."""
    B = image_all.shape[0]
    full_i = logit_scale * (image_all @ text_all.T)
    full_t = logit_scale * (text_all @ image_all.T)
    logits_i, logits_t = full_i[rows], full_t[rows]
    b = logits_i.shape[0]
    ar = torch.arange(b)
    labels = ar + rows.start
    dissim = _dissim_rows(dino_all, rows)

    beta_i = _beta(full_i, rho, c_clip)
    tilde_i, delta_i, rhat_i, p_i = _shift(logits_i, dissim, beta_i, c_clip, rows)
    if text_sym:
        beta_t = _beta(full_t, rho, c_clip)
        tilde_t, delta_t, rhat_t, p_t = _shift(logits_t, dissim, beta_t, c_clip, rows)
    else:
        tilde_t, delta_t, rhat_t, p_t, beta_t = logits_t, None, None, None, None
    ce_i = F.cross_entropy(tilde_i, labels)
    ce_t = F.cross_entropy(tilde_t, labels)
    loss = 0.5 * (ce_i + ce_t)

    with torch.no_grad():
        zero = torch.zeros((), dtype=image_all.dtype)
        off = float(b * B - b)

        def side(delta, r_hat, p_base, tilde):
            if delta is None:
                return dict(pc=zero, dmax=zero, dmean=zero, dstd=zero, diag=zero, corr=zero, pos=zero)
            p_mod = torch.softmax(tilde, dim=1)
            d_abs = delta.abs()
            diag = r_hat[ar, labels]
            pos = ((r_hat > 0).float().sum() - (diag > 0).float().sum()) / off
            return dict(pc=(p_base * r_hat).sum(dim=1).abs().mean(), dmax=d_abs.max(), dmean=d_abs.mean(),
                        dstd=d_abs.std(), diag=diag.abs().max(), corr=row_corr_mean(r_hat, p_mod - p_base), pos=pos)

        si = side(delta_i, rhat_i, p_i.detach(), tilde_i.detach())
        st = side(delta_t, rhat_t, None if p_t is None else p_t.detach(), tilde_t.detach())
        p_t_base = torch.softmax(logits_t.detach(), dim=1)
        dbg = {
            "pc_err_img": si["pc"], "pc_err_txt": st["pc"],
            "diag_max_img": si["diag"], "diag_max_txt": st["diag"],
            "delta_img_max": si["dmax"], "delta_img_mean": si["dmean"], "delta_img_std": si["dstd"],
            "delta_txt_max": st["dmax"], "delta_txt_mean": st["dmean"], "delta_txt_std": st["dstd"],
            "l1_prob_shift_img": (torch.softmax(tilde_i.detach(), dim=1) - p_i.detach()).abs().sum(dim=1).mean(),
            "l1_prob_shift_txt": (torch.softmax(tilde_t.detach(), dim=1) - p_t_base).abs().sum(dim=1).mean(),
            "corr_rhat_dprob_img": si["corr"], "corr_rhat_dprob_txt": st["corr"],
            "ce_img_base": F.cross_entropy(logits_i.detach(), labels),
            "ce_txt_base": F.cross_entropy(logits_t.detach(), labels),
            "ce_img_mod": ce_i.detach(), "ce_txt_mod": ce_t.detach(),
            "pos_frac_img": si["pos"], "neg_frac_img": 1.0 - si["pos"],
            "pos_frac_txt": st["pos"], "neg_frac_txt": (1.0 - st["pos"]) if text_sym else zero,
            "beta_img": beta_i, "beta_txt": beta_t if text_sym else zero,
            "rho": rho, "clip_c": c_clip,
        }
    return loss, dbg
