"""L2-bounded NB / tar-NB without a GPU: the CPU reference the GPU tests compare with (tests/l2_reference.py) against an
fp64 numpy restatement of torchattacks PGDL2's step and per-block projection on a small differentiable model, and the attack
classes' handling of the ``norm`` argument."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))      # tests/l2_reference.py
import l2_reference as R  # noqa: E402

K = 5          # classes of the toy model


class _Linear:
    """logp = log_softmax(W x + b) point by point: a model whose input gradient has a closed form."""

    def __init__(self, seed, colour_weight=1.0):
        g = np.random.default_rng(seed)
        self.W = g.normal(0, 1, (K, 9))
        self.W[:, 3:6] *= colour_weight
        self.b = g.normal(0, 0.1, K)

    def __call__(self, x):
        z = torch.einsum("kc,bcn->bnk", torch.from_numpy(self.W).float(), x) + torch.from_numpy(self.b).float()
        return torch.log_softmax(z, 2), None

    def grad(self, x, y, scale):
        """d(scale * sum CE(y)) / dx on the colour channels, fp64."""
        z = np.einsum("kc,bcn->bnk", self.W, x) + self.b
        p = np.exp(z - z.max(2, keepdims=True))
        p /= p.sum(2, keepdims=True)
        p[np.arange(x.shape[0])[:, None], np.arange(x.shape[2])[None, :], y] -= 1.0
        return scale * np.einsum("bnk,kc->bcn", p, self.W)[:, 3:6]


def _np_attack(model, x, y, eps, alpha, iters, sign, scale, mask=None):
    """fp64 restatement: returns the un-projected last step and the projected colours entering every step."""
    x = x.astype(np.float64)
    B, _, N = x.shape
    mv = np.ones((B, 1, N), bool) if mask is None else mask.reshape(B, 1, N)
    ori = x[:, 3:6].copy()
    col = ori.copy()
    adv = x.copy()
    cols = []
    for _ in range(iters):
        cols.append(col.copy())
        xin = x.copy()
        xin[:, 3:6] = np.where(mv, col, x[:, 3:6])
        g = model.grad(xin, y, scale) * mv
        gn = np.sqrt((g ** 2).reshape(B, -1).sum(1)).reshape(B, 1, 1)
        a = col + sign * alpha * g / (gn + 1e-10)
        d = (a - ori) * mv
        dn = np.sqrt((d ** 2).reshape(B, -1).sum(1)).reshape(B, 1, 1)
        f = np.where(dn > eps, eps / np.where(dn > 0, dn, 1.0), 1.0)
        adv[:, 3:6] = np.where(mv, a, adv[:, 3:6])
        col = np.clip(ori + d * f, 0, 1)
    return adv, cols


def _data(B, N, seed):
    g = np.random.default_rng(seed)
    x = g.uniform(0, 1, (B, 9, N)).astype(np.float32)
    y = g.integers(0, K, (B, N))
    return x, y


@pytest.mark.parametrize("eps, alpha", [(0.05, 0.2), (2.0, 0.1)], ids=["projection_fires", "inside_the_ball"])
def test_nb_l2_oracle_matches_fp64(eps, alpha):
    model = _Linear(0)
    x, y = _data(3, 64, 1)
    snaps = []
    got = R.nb_attack_l2(model, torch.from_numpy(x), y.astype(np.float64), eps=eps, alpha=alpha, iters=4, snapshots=snaps)
    want, cols = _np_attack(model, x, y, eps, alpha, 4, +1.0, 1.0 / 64)
    np.testing.assert_allclose(got.numpy(), want, rtol=0, atol=2e-6)
    for s, c in zip(snaps, cols):
        np.testing.assert_allclose(s.numpy(), c, rtol=0, atol=2e-6)
    dcol = np.sqrt(((cols[-1] - x[:, 3:6]) ** 2).reshape(3, -1).sum(1))
    if alpha > eps:
        # every block was projected onto the sphere; the clamp to [0, 1] after the projection can only shorten it
        assert (dcol <= eps * (1 + 1e-6)).all() and dcol.max() > eps * (1 - 1e-6)
    else:
        assert (dcol < eps).all()
    # Q1: the returned tensor is the un-projected last step, within eps + alpha of the input, not within eps
    dadv = np.sqrt(((got.numpy() - x)[:, 3:6] ** 2).reshape(3, -1).sum(1))
    assert (dadv <= eps + alpha + 1e-5).all()
    if alpha > eps:
        assert (dadv > eps + 1e-3).all()
    assert torch.equal(got[:, :3], torch.from_numpy(x[:, :3])) and torch.equal(got[:, 6:], torch.from_numpy(x[:, 6:]))


def test_tar_nb_l2_oracle_matches_fp64_with_an_all_zero_mask_row():
    model = _Linear(2)
    B, N = 3, 48
    x, _ = _data(B, N, 3)
    mask = np.random.default_rng(4).uniform(size=(B, N)) < 0.4
    mask[1] = False
    got = R.tar_nb_attack_l2(model, torch.from_numpy(x), eps=0.08, alpha=0.05, iters=5, target=2, mask=torch.from_numpy(mask))
    want, _ = _np_attack(model, x, np.full((B, N), 2), 0.08, 0.05, 5, -1.0, 1.0 / (B * N), mask)
    np.testing.assert_allclose(got.numpy(), want, rtol=0, atol=2e-6)
    assert torch.equal(got[1], torch.from_numpy(x[1]))                                  # nothing moves in the empty block
    m3 = np.broadcast_to(mask[:, None], (B, 3, N))
    assert np.array_equal(got.numpy()[:, 3:6][~m3], x[:, 3:6][~m3])                     # unmasked colours untouched
    assert not torch.isnan(got).any()


def test_nb_l2_zero_gradient_leaves_the_input():
    model = _Linear(5, colour_weight=0.0)       # no colour dependence: g = 0 on every block
    x, y = _data(2, 32, 6)
    got = R.nb_attack_l2(model, torch.from_numpy(x), y.astype(np.float64), eps=0.1, alpha=0.05, iters=3)
    assert torch.equal(got, torch.from_numpy(x))


def test_l2_step_is_separately_rounded_fp32_in_the_kernel_order():
    """Given its two norms, the step is the fp32 op sequence of pgd_l2_update_kernel, bit for bit."""
    g = np.random.default_rng(9)
    B, N = 3, 40
    col = g.uniform(0, 1, (B, 3, N)).astype(np.float32)
    ori = np.clip(col + g.normal(0, 0.2, col.shape), 0, 1).astype(np.float32)
    grad = (g.normal(0, 1e-8, col.shape)).astype(np.float32)
    moving = g.uniform(size=(B, 1, N)) < 0.5
    alpha, eps = np.float32(-0.3), np.float32(0.4)
    a, c = R.l2_step(torch.from_numpy(col), torch.from_numpy(ori), torch.from_numpy(grad), float(alpha), float(eps),
                     torch.from_numpy(moving))
    f32 = np.float32
    for b in range(B):
        m = np.broadcast_to(moving[b], (3, N))
        gn = f32(np.sqrt((grad[b][m].astype(np.float64) ** 2).sum()))
        ab = col[b] + alpha * (grad[b] / (gn + f32(1e-10)))
        d = ab - ori[b]
        dn = f32(np.sqrt((d[m].astype(np.float64) ** 2).sum()))
        fb = eps / dn if dn > eps else f32(1.0)
        cb = np.clip(ori[b] + d * fb, f32(0), f32(1))
        assert ab.dtype == np.float32 and cb.dtype == np.float32
        assert np.array_equal(a[b].numpy()[m], ab[m]) and np.array_equal(c[b].numpy()[m], cb[m])


def test_attack_classes_take_the_norm():
    from pointsecguard_b200 import torchattacks
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    m = get_model(13)
    for cls in (torchattacks.NB_attack, torchattacks.tar_NB_attack):
        with pytest.raises(ValueError):
            cls(m, norm="L1")
        with pytest.raises(ValueError):
            cls(m, norm="l2")
    head = "model_name=get_model, training=True, device=cpu, eps=0.3, alpha=0.00784313725490196, iters=40, "
    assert str(torchattacks.NB_attack(m)) == "NB_attack(" + head + "attack_mode=default, return_type=float)"
    assert str(torchattacks.tar_NB_attack(m)) == ("tar_NB_attack(" + head + "target=None, mask=None, attack_mode=default, "
                                                  "return_type=float)")
    assert str(torchattacks.NB_attack(m, norm="Linf")) == str(torchattacks.NB_attack(m))
    s = str(torchattacks.NB_attack(m, eps=1.0, norm="L2"))
    assert s.startswith("NB_attack(model_name=get_model") and "eps=1.0" in s and s.endswith(", norm=L2)")
    assert str(torchattacks.tar_NB_attack(m, target=7, norm="L2")).endswith("return_type=float, norm=L2)")
