"""fp64 statement of open_clip's SigLipLoss (2.31.0, as the fork carries it) for the SigLIP tests.

No golden fixture of the reference exists for this loss: the reference tree is not available where the fixtures are
made.  This file restates the upstream recipe instead - the +-1 labels matrix, `-logsigmoid(labels * logits).sum() / n`
on the local block, plus the neighbour blocks with negative labels only - and is pinned two other ways:
tests/test_siglip_host.py runs the upstream `gather` recipe as a W-process gloo job (torch.distributed.nn.all_gather)
and compares its per-rank losses and gradients with `rank_grads`, and runs the staged reference's own SigLipLoss for
every dist_impl when oracle/_ref/loss.py exists.

Convention (as the module): features get the derivative of the SUM of all ranks' losses, logit_scale / logit_bias
that of rank r's own loss."""
import torch
import torch.nn.functional as F


def block_loss(img, txt, scale, bias, negative_only=False):
    """Upstream `SigLipLoss._loss`: one [n x n] block, n = img rows."""
    logits = scale * img @ txt.T
    if bias is not None:
        logits = logits + bias
    n = img.shape[0]
    labels = -torch.ones((n, n), dtype=img.dtype, device=img.device)
    if not negative_only:
        labels = 2 * torch.eye(n, dtype=img.dtype, device=img.device) + labels
    return -F.logsigmoid(labels * logits).sum() / n


def rank_loss(img_all, txt_all, scale, bias, world, r):
    """Rank r's loss on the concatenated batch: its own block, then every other rank's captions as negatives."""
    b = img_all.shape[0] // world
    im = img_all[r * b:(r + 1) * b]
    loss = block_loss(im, txt_all[r * b:(r + 1) * b], scale, bias)
    for i in range(world):
        if i != r:
            loss = loss + block_loss(im, txt_all[i * b:(i + 1) * b], scale, bias, negative_only=True)
    return loss


def rank_grads(img, txt, scale, bias, world):
    """Per rank: loss, d_image / d_text rows (of the sum of all ranks' losses), d_scale / d_bias (own loss)."""
    dt = torch.float64
    im = img.to(dt).clone().requires_grad_(True)
    tx = txt.to(dt).clone().requires_grad_(True)
    sc = torch.tensor(float(scale), dtype=dt, device=img.device, requires_grad=True)
    bi = None if bias is None else torch.tensor(float(bias), dtype=dt, device=img.device, requires_grad=True)
    per = [rank_loss(im, tx, sc, bi, world, r) for r in range(world)]
    own = []
    for p in per:
        g = torch.autograd.grad(p, [sc] if bi is None else [sc, bi], retain_graph=True)
        own.append((float(g[0]), None if bi is None else float(g[1])))
    sum(per).backward()
    b = img.shape[0] // world
    return [dict(loss=float(per[r].detach()), d_image=im.grad[r * b:(r + 1) * b], d_text=tx.grad[r * b:(r + 1) * b],
                 d_scale=own[r][0], d_bias=own[r][1]) for r in range(world)]


def blocked(img, txt, scale, bias, rows=(), cols=(), block=2048):
    """World size 1 in fp64 row blocks, never more than [block x B]: the loss, d_scale, d_bias, and d_image / d_text
    of the given row blocks (lists of slices).  For batches whose B x B fp64 logits do not fit."""
    B = img.shape[0]
    I, T = img.double(), txt.double()
    loss = ds = db = 0.0
    for r0 in range(0, B, block):
        z = scale * I[r0:r0 + block] @ T.T + (0.0 if bias is None else bias)
        lab = -torch.ones_like(z)
        idx = torch.arange(r0, min(r0 + block, B), device=z.device)
        lab[idx - r0, idx] = 1.0
        loss += float(F.softplus(-lab * z).sum())
        g = -lab * torch.sigmoid(-lab * z)
        ds += float((g * (z - (0.0 if bias is None else bias)) / scale).sum())
        db += float(g.sum())
    out = dict(loss=loss / B, d_scale=ds / B, d_bias=db / B, d_image=[], d_text=[])

    def gblock(zr, zc):  # G of rows zr x columns zc
        z = scale * I[zr] @ T[zc].T + (0.0 if bias is None else bias)
        ri = torch.arange(B, device=z.device)[zr][:, None]
        ci = torch.arange(B, device=z.device)[zc][None, :]
        lab = torch.where(ri == ci, 1.0, -1.0).to(z.dtype)
        return -lab * torch.sigmoid(-lab * z)

    for sl in rows:
        out["d_image"].append(sum(scale / B * gblock(sl, slice(c, c + block)) @ T[c:c + block]
                                  for c in range(0, B, block)))
    for sl in cols:
        out["d_text"].append(sum(scale / B * gblock(slice(r, r + block), sl).T @ I[r:r + block]
                                 for r in range(0, B, block)))
    return out
