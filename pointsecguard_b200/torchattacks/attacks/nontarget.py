"""Non-targeted colour attacks -- drop-in for PointNet/attacks/torchattacks/attacks/nontarget.py.

NB_attack (:10-42): L-inf sign ascent on sum-CE / N over channels 3:6; the returned tensor is the
un-projected last step (Q1).  ``norm="L2"`` replaces the sign step and box projection by torchattacks PGDL2's
normalised-gradient step and per-block L2-ball projection (eps is then the radius of the ball).  The whole loop is one C call (psg_nb_attack): the geometry of all
``iters`` forwards is computed in one batched pass first, because for a colour attack it depends
only on xyz and on the FPS start draws (made here on the CPU generator in the reference's order).
"""
from __future__ import annotations

import torch

from ..attack import Attack

_MAX_PROBLEMS = 1024     # FPS problems (= forwards x blocks) whose geometry is resident at once
NORMS = ("Linf", "L2")


def _check_norm(norm):
    if norm not in NORMS:
        raise ValueError(f"norm must be one of {NORMS}, got {norm!r}")
    return norm


def _str_with_norm(s, norm):
    """The string form of the reference's attacks, with the norm listed when it is not the reference's L-inf."""
    return s if norm == "Linf" else s[:-1] + f", norm={norm})"


class NB_attack(Attack):
    def __init__(self, model, eps=0.3, alpha=2 / 255, iters=40, norm="Linf"):
        super().__init__("NB_attack", model)
        self.eps = eps
        self.alpha = alpha
        self.iters = iters
        self._norm = _check_norm(norm)

    def __str__(self):
        return _str_with_norm(super().__str__(), self._norm)

    def forward(self, images, labels):
        return _nb_loop(self, images, labels, target=-1, mask=None)


def _head_start(model, t):
    """Forwards of a geometry chunk that run on the primary engine while the rest of the chunk's geometry is computed
    on a side stream (0 = no pipelining).  ``model.geometry_head`` overrides the default of 4 (measured at B = 16: 20 iterations 14.55 -> 14.14 ms, 50 iterations 34.0 -> 33.75 ms)."""
    want = int(getattr(model, "geometry_head", 4))
    if want <= 0 or t < 4 * want:
        return 0
    return want


def _nb_loop(atk, images, labels, target, mask):
    eng = atk._engine(images)
    dev = images.device
    B, C, N = images.shape
    src = images.detach()
    norm = atk._norm
    # nontarget.py:34: sum-CE / N;  target.py:38: mean CE over the B*N points.  The sign step ignores the scale; the L2
    # step does not (the 1e-10 beside the gradient norm), so there the mean runs over the GLOBAL batch: a shard's blocks
    # then step exactly as they do in the single-GPU run.
    if target < 0:
        scale = 1.0 / N
    elif norm == "L2":
        scale = 1.0 / ((eng.shard.global_batch if eng.shard is not None else B) * N)
    else:
        scale = 1.0 / (B * N)
    chunk = max(1, min(atk.iters, _MAX_PROBLEMS // B))
    cur = torch.cuda.current_stream()
    eng.use_stream(None)                            # on `cur`: the head start's events order the tail engine against it
    eng.bind(B, N, chunk)
    eng.set_xyz_grad(False)                         # colour attack: no geometric gradient (decided before the geometry pass)
    eng.set_input(src)
    adv = ori = lab = msk = None
    done = 0
    while done < atk.iters:
        t = min(chunk, atk.iters - done)
        starts = eng.draw_starts(t)                                     # int32 [4, t, B]
        # Head start: the geometry pass is a latency chain (1360 dependent FPS rounds) whatever the number of forwards, so
        # the first `head` forwards get their own small pass on the primary engine and the loop starts on them, while a
        # second engine (own workspace, side stream) computes the geometry of the remaining forwards beside those first
        # steps.  Same draws, same kernels, same values: results are bit-identical.
        head = _head_start(atk.model, t)
        tail = tail_ready = None
        if head:
            tail, side = atk.model.tail_engine(dev, eng)
            tail.bind(B, N, t - head)
            tail.set_xyz_grad(False)
            fork = torch.cuda.Event()
            fork.record(cur)
            side.wait_event(fork)
            tail.use_stream(side)
            try:
                tail.set_input(src)
                tail.geometry(starts[:, head:].contiguous())
                tail_ready = torch.cuda.Event()
                tail_ready.record(side)
            finally:
                tail.use_stream(None)
            eng.geometry(starts[:, :head].contiguous())
        else:
            eng.geometry(starts)
        if adv is None:
            # the loop's own tensors are made AFTER the first geometry pass is enqueued: their host work (label / mask
            # conversion and upload, clones) then runs while the GPU computes FPS / ball query / 3-NN instead of before it
            adv = images.detach().clone(memory_format=torch.contiguous_format)
            ori = images.detach()[:, 3:6].contiguous()
            lab = atk._labels_i32(labels, dev) if target < 0 else None
            msk = atk._mask_u8(mask, B, N, dev) if mask is not None else None
            if msk is not None and B > 1 and getattr(mask, "ndim", 2) == 1:
                # target.py:26,36 with a batch: the cost reads outputs[0] only, so the gradient of every other block is
                # zero and sign(0) = 0 leaves it where it is -- the reference attacks block 0 alone.  A [B,N] mask
                # attacks every block.
                msk = msk.clone()
                msk[1:] = 0
        if head:
            for i in range(head):
                eng.nb_attack(adv, ori, msk, lab, target, 1, i, atk.alpha, atk.eps, scale, norm)
            cur.wait_event(tail_ready)
            tail.copy_input_from(eng)          # the PROJECTED colours of the head's last update (adv holds the un-projected ones)
            for i in range(t - head):
                tail.nb_attack(adv, ori, msk, lab, target, 1, i, atk.alpha, atk.eps, scale, norm)
            if done + t < atk.iters:
                eng.copy_input_from(tail)      # the next chunk starts on the primary engine again
        else:
            for i in range(t):
                eng.nb_attack(adv, ori, msk, lab, target, 1, i, atk.alpha, atk.eps, scale, norm)
        done += t
    if adv is None:                                                        # iters == 0
        adv = images.detach().clone(memory_format=torch.contiguous_format)
    atk.model._generation += 1
    return adv


class NU_attack(Attack):
    """nontarget.py:44-135.  ``field`` / ``box`` are extensions (default = the reference: colours 3:6 in
    [0,1]): ``field=(0, 6)`` perturbs coordinates and colours (BASELINE.json configs[2])."""

    def __init__(self, model, c=1e-4, kappa=0, steps=1000, lr=0.01, field=None, box=None):
        super().__init__("NU_attack", model)
        self.c = c
        self.kappa = kappa
        self.steps = steps
        self.lr = lr
        self.field = field
        self.box = box

    def forward(self, images, labels):
        from pointsecguard_b200 import nu
        return nu.nu_attack(self, images, labels, mask=None, target=None, neighbour=10)
