"""Targeted / masked colour attacks -- drop-in for PointNet/attacks/torchattacks/attacks/target.py.

tar_NB_attack (:7-45): sign *descent* on the mean CE to ``target`` over all points, only masked
points' colours move (unmasked points are neither stepped nor clamped, target.py:41-43).  The reference handles
B == 1 with a [N] mask; handed a batch it still attacks block 0 only (its cost reads ``outputs[0]``, :36), and so does
this class for a 1-D mask.  A [B,N] mask is the generalisation to batches (SURVEY.md section 8c) with identical
per-block arithmetic (the step is a sign, so the loss normalisation does not matter).  ``norm="L2"`` takes torchattacks
PGDL2's step and per-block L2-ball projection over the masked points instead (nontarget.py, _nb_loop).
"""
from __future__ import annotations

from ..attack import Attack
from .nontarget import _check_norm, _nb_loop, _str_with_norm


class tar_NB_attack(Attack):
    def __init__(self, model, eps=0.3, alpha=2 / 255, iters=40, target=None, mask=None, norm="Linf"):
        super().__init__("tar_NB_attack", model)
        self.eps = eps
        self.alpha = alpha
        self.iters = iters
        self.target = target
        self.mask = mask
        self._norm = _check_norm(norm)

    def __str__(self):
        return _str_with_norm(super().__str__(), self._norm)

    def forward(self, images, labels):
        if self.target is None or self.mask is None:
            raise ValueError("tar_NB_attack needs target and mask (target.py:8)")
        return _nb_loop(self, images, labels, target=int(self.target), mask=self.mask)


class tar_NU_attack(Attack):
    def __init__(self, model, c=1e-4, kappa=0, steps=1000, lr=0.01, target=None, mask=None):
        super().__init__("tar_NU_attack", model)
        self.c = c
        self.kappa = kappa
        self.steps = steps
        self.lr = lr
        self.target = target
        self.mask = mask

    def forward(self, images, labels):
        from pointsecguard_b200 import nu
        return nu.nu_attack(self, images, labels, mask=self.mask, target=self.target, neighbour=5)
