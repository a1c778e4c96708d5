"""fp64 statement of open_clip's DistillClipLoss (2.31.0) with local_loss for the DistillClipLoss tests.

No golden fixture of the reference exists for this loss.  This file restates the upstream recipe - student and
teacher logits of this rank's rows against all B columns (`gather_features` + `get_logits` with local_loss), CE with
the global diagonal labels, and `-(softmax(teacher) * log_softmax(student)).sum(1).mean(0)` per direction - and is
pinned by tests/test_distill_host.py against that recipe run as a W-process gloo job (and against the staged
reference's own class when oracle/_ref/loss.py exists).

Convention (as the module): with upstream gradients g_c, g_d of the two losses, the features get the derivative of
sum_r (g_c contrastive_r + g_d distill_r) with respect to rank r's rows (gather_with_grad=False: of rank r's own
losses, the gathered copies being constants), logit_scale that of rank r's own losses.  The teacher gets nothing."""
import torch
import torch.nn.functional as F


def _dist(teacher, student):
    return -(teacher.softmax(dim=1) * student.log_softmax(dim=1)).sum(dim=1).mean(dim=0)


def rank_losses(im_rows, tx_rows, im_cols, tx_cols, dim_rows, dtx_rows, dim_cols, dtx_cols, s, st, r):
    """Rank r's (contrastive, distill): rows are its b images / texts, columns all B of the other modality."""
    b = im_rows.shape[0]
    lpi, lpt = s * im_rows @ tx_cols.T, s * tx_rows @ im_cols.T
    dpi, dpt = st * dim_rows @ dtx_cols.T, st * dtx_rows @ dim_cols.T
    labels = torch.arange(b, device=im_rows.device) + r * b
    contrastive = (F.cross_entropy(lpi, labels) + F.cross_entropy(lpt, labels)) / 2
    distill = (_dist(dpi, lpi) + _dist(dpt, lpt)) / 2
    return contrastive, distill


def rank_grads(img, txt, dimg, dtxt, s, st, world, gather_with_grad=True, gc=1.0, gd=1.0):
    """Per rank: both losses, d_image / d_text rows, d_scale (own losses), for upstream gradients gc, gd."""
    dt = torch.float64
    im = img.to(dt).clone().requires_grad_(True)
    tx = txt.to(dt).clone().requires_grad_(True)
    di, dx = dimg.to(dt), dtxt.to(dt)
    b = img.shape[0] // world
    out = []
    total = 0.0
    for r in range(world):
        sl = slice(r * b, (r + 1) * b)
        sc = torch.tensor(float(s), dtype=dt, device=img.device, requires_grad=True)
        cols_i, cols_t = (im, tx) if gather_with_grad else (im.detach(), tx.detach())
        c, d = rank_losses(im[sl], tx[sl], cols_i, cols_t, di[sl], dx[sl], di, dx, sc, float(st), r)
        own = gc * c + gd * d
        (g_s,) = torch.autograd.grad(own, [sc], retain_graph=True)
        out.append(dict(contrastive=float(c.detach()), distill=float(d.detach()), d_scale=float(g_s)))
        total = total + own
    total.backward()
    for r in range(world):
        out[r]["d_image"] = im.grad[r * b:(r + 1) * b]
        out[r]["d_text"] = tx.grad[r * b:(r + 1) * b]
    return out


def blocked(img, txt, dimg, dtxt, s, st, gc=1.0, gd=1.0, rows=(), cols=(), block=2048):
    """World size 1 in fp64 row blocks, never more than [block x B] at a time: both losses, d_scale, and d_image /
    d_text of the given row slices.  For batches whose B x B fp64 logits do not fit."""
    B = img.shape[0]
    I, T, DI, DT = img.double(), txt.double(), dimg.double(), dtxt.double()
    stats = {}
    out = dict(contrastive=0.0, distill=0.0)
    for name, (A, Bm, DA, DB) in (("i", (I, T, DI, DT)), ("t", (T, I, DT, DI))):
        lse, lset = [], []
        for r0 in range(0, B, block):
            x, t = s * A[r0:r0 + block] @ Bm.T, st * DA[r0:r0 + block] @ DB.T
            lx, lt = torch.logsumexp(x, 1), torch.logsumexp(t, 1)
            idx = torch.arange(r0, min(r0 + block, B), device=x.device)
            out["contrastive"] += float((lx - x[idx - r0, idx]).sum()) / (2 * B)
            out["distill"] += float((lx - ((t - lt[:, None]).exp() * x).sum(1)).sum()) / (2 * B)
            lse.append(lx)
            lset.append(lt)
        stats[name] = (torch.cat(lse), torch.cat(lset))

    def dl(rs, cs):  # dL/dx of image rows rs x text columns cs
        x, t = s * I[rs] @ T[cs].T, st * DI[rs] @ DT[cs].T
        pr, qr = (x - stats["i"][0][rs, None]).exp(), (t - stats["i"][1][rs, None]).exp()
        pc, qc = (x - stats["t"][0][None, cs]).exp(), (t - stats["t"][1][None, cs]).exp()
        g = (gc + gd) * (pr + pc) - gd * (qr + qc)
        ri = torch.arange(B, device=x.device)[rs][:, None]
        ci = torch.arange(B, device=x.device)[cs][None, :]
        g = g - 2 * gc * (ri == ci).to(g.dtype)
        return g / (2 * B), x

    ds = 0.0
    for r0 in range(0, B, block):
        g, x = dl(slice(r0, r0 + block), slice(0, B))
        ds += float((g * x).sum()) / s
    out["d_scale"] = ds
    out["d_image"] = [sum(s * dl(sl, slice(c, c + block))[0] @ T[c:c + block] for c in range(0, B, block))
                      for sl in rows]
    out["d_text"] = [sum(s * dl(slice(r, r + block), sl)[0].T @ I[r:r + block] for r in range(0, B, block))
                     for sl in cols]
    return out
