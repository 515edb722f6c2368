"""CPU reference of the L2-bounded NB / tar-NB attacks (torchattacks PGDL2's step and per-block L2-ball projection), for
the tests of ``norm="L2"``.  The loops are those of oracle/attacks_oracle.py (nb_attack :32-51, tar_nb_attack :54-79: the
reference's nontarget.py:28-39 / target.py:31-43) with only the update replaced by ``l2_step``; model calls, costs and FPS
draws are the same, so a run with the same seed sees the same geometry as the package's attack."""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from oracle.attacks_oracle import _labels


def l2_step(col, ori, g, alpha_signed, eps, moving=None):
    """One step per block over the entries where ``moving`` (bool, broadcast to g) holds:
    gn = fp32(sqrt(sum double(g)^2)), a = col + alpha_signed * (g / (gn + 1e-10)), d = a - ori,
    dn = fp32(sqrt(sum double(d)^2)), f = eps / dn if dn > eps else 1.  Returns (a, clamp(ori + d * f, 0, 1)); every
    element op is one fp32 op in that order, as in csrc/elementwise.cu (pgd_l2_update_kernel)."""
    f32 = lambda v: torch.tensor(v, dtype=torch.float32)

    def norm(v):
        v = v if moving is None else torch.where(moving, v, torch.zeros_like(v))
        return v.double().pow(2).flatten(1).sum(1).sqrt().float().view(-1, *([1] * (v.dim() - 1)))

    a = col + f32(alpha_signed) * (g / (norm(g) + f32(1e-10)))
    d = a - ori
    dn = norm(d)
    f = torch.where(dn > f32(eps), f32(eps) / dn, f32(1.0))
    return a, torch.clamp(ori + d * f, 0, 1)


def nb_attack_l2(model, images, labels, eps, alpha, iters, snapshots=None):
    """Ascent on sum-CE / N with the L2 step on colours 3:6; returns the un-projected last step (Q1).
    ``snapshots``: optional list that receives the projected colours entering every iteration."""
    col = images[:, 3:6].clone().detach()
    ori = col.clone()
    adv = images.clone().detach()
    y = _labels(labels).to(images.device)
    for _ in range(iters):
        if snapshots is not None:
            snapshots.append(col.detach().clone())
        col.requires_grad_(True)
        adv[:, 3:6] = col
        logp, _ = model(adv)
        cost = F.cross_entropy(logp.reshape(-1, logp.size(2)), y.view(-1), reduction="sum") / logp.size(1)
        g, = torch.autograd.grad(cost, col)
        adv = adv.detach()
        adv[:, 3:6], col = l2_step(col.detach(), ori, g, alpha, eps)
    return adv


def tar_nb_attack_l2(model, images, eps, alpha, iters, target, mask, snapshots=None):
    """Descent on the mean CE to ``target`` over all B*N points with the L2 step over the masked points of each block.
    mask: bool [N] (every block) or [B,N]."""
    m = torch.as_tensor(np.asarray(mask)) if not torch.is_tensor(mask) else mask
    B, _, N = images.shape
    m = m.view(1, N).expand(B, N) if m.dim() == 1 else m
    m3 = m.view(B, 1, N)
    col = images[:, 3:6].clone().detach()
    ori = col.clone()
    adv = images.clone().detach()
    tgt = torch.full((B * N,), int(target), dtype=torch.int64)
    for _ in range(iters):
        if snapshots is not None:
            snapshots.append(col.detach().clone())
        col.requires_grad_(True)
        adv[:, 3:6] = torch.where(m3, col, adv[:, 3:6])
        logp, _ = model(adv)
        cost = F.cross_entropy(logp.reshape(-1, logp.size(2)), tgt)
        g, = torch.autograd.grad(cost, col)
        adv = adv.detach()
        stepped, col = l2_step(col.detach(), ori, g, -alpha, eps, m3)
        adv[:, 3:6] = torch.where(m3, stepped, adv[:, 3:6])
    return adv
