"""TF32-exact reference of the engine's network (TEST INFRASTRUCTURE ONLY; see oracle/__init__.py).

The tcgen05 TF32 mode (engine.MLP_TF32) is fully determined arithmetic:

  * every layer's weights are rounded on the host to nearest TF32 after the truncation compensation,
    ``tf32_rna(w * (1 + 3.45e-4))`` (csrc/net.cu: psg_mlp_create); layers loaded on the device round
    ``w * (1.f + 3.45e-4f)`` taken in fp32 the same way (csrc/train.cu: repack_kernel);
  * ``tcgen05.mma.kind::tf32`` truncates each fp32 operand to its top 19 bits, so the activations (forward)
    and the pre-activation gradients (dgrad) enter every product truncated;
  * products accumulate in fp32, and everything else -- bias, ReLU, max-pool, interpolation, segmented sums,
    the loss gradient -- is fp32 on the CUDA cores.

This module applies exactly those two roundings inside an fp64 computation, so it differs from the kernels
only by fp32 summation order (and the accumulator's own truncation, ~2e-9 K relative per layer).  With
``tf32=False`` the same walk is the plain fp64 reference of the fp32 and 3xTF32 modes.

The network walk consumes the folded weights of ``model.describe()`` (engine column order: the first SA
layer reads ``[features | xyz - centre]``, FP layers ``[skip | interp]``, MSG branches concatenated in
order) and the geometry the engine computed (``Engine.read_geometry``), so only the numerics are compared.
It runs on any device in float64; on a GPU, plain fp64 matmuls do not use TF32.
"""
from __future__ import annotations

import numpy as np
import torch

TF32_COMP = 3.45e-4                                         # csrc/net.cu kTf32Comp
_COMP_F32 = float(np.float32(1.0) + np.float32(TF32_COMP))  # repack_kernel: 1.f + (float)comp, in fp32


def _bits(f32: torch.Tensor) -> torch.Tensor:
    return f32.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF


def _from_bits(u: torch.Tensor) -> torch.Tensor:
    u = torch.where(u >= 2 ** 31, u - 2 ** 32, u)
    return u.to(torch.int32).view(torch.float32)


def tf32_rna(x: torch.Tensor) -> torch.Tensor:
    """csrc/net.cu tf32_rna: round to fp32 (nearest even), then to nearest TF32 with ties away from zero
    (``(u + 0x1000) & 0xffffe000``); Inf and NaN pass unchanged.  Returns float32."""
    f = x.to(torch.float32)
    u = _bits(f)
    special = (u & 0x7F800000) == 0x7F800000
    return torch.where(special, f, _from_bits((u + 0x1000) & 0xFFFFE000))


def tf32_rna_host_weights(w) -> torch.Tensor:
    """The host-side weight rounding of psg_mlp_create: product with (1 + 3.45e-4) taken in double."""
    return tf32_rna(torch.as_tensor(w).to(torch.float64) * (1.0 + TF32_COMP))


def tf32_rna_device_weights(w) -> torch.Tensor:
    """repack_kernel's rounding: ``v * (1.f + comp)`` in fp32, then the same bit rounding (no Inf/NaN test there,
    which matters only for non-finite weights)."""
    f = torch.as_tensor(w).to(torch.float32) * torch.tensor(_COMP_F32, dtype=torch.float32)
    return _from_bits((_bits(f) + 0x1000) & 0xFFFFE000)


def tf32_trunc(x: torch.Tensor) -> torch.Tensor:
    """What tcgen05.mma kind::tf32 reads of an fp32 operand: the top 19 bits (``u & 0xffffe000``).  Returns float32."""
    return _from_bits(_bits(x.to(torch.float32)) & 0xFFFFE000)


class _Linear(torch.autograd.Function):
    """y = A W^T + b.  TF32 mode: A truncated before the product, the result rounded to fp32; the dgrad takes the
    pre-activation gradient truncated, dA = trunc(dY) W, rounded to fp32.  Plain mode: exact fp64 both ways."""

    @staticmethod
    def forward(ctx, a, w, b, tf32):
        ctx.save_for_backward(w)
        ctx.tf32 = tf32
        if tf32:
            a = tf32_trunc(a).to(w.dtype)
        y = torch.addmm(b, a.reshape(-1, a.shape[-1]), w.t()).reshape(*a.shape[:-1], w.shape[0])
        return y.float().to(w.dtype) if tf32 else y

    @staticmethod
    def backward(ctx, dy):
        (w,) = ctx.saved_tensors
        if ctx.tf32:
            dy = tf32_trunc(dy).to(w.dtype)
        da = (dy.reshape(-1, dy.shape[-1]) @ w).reshape(*dy.shape[:-1], w.shape[1])
        return (da.float().to(w.dtype) if ctx.tf32 else da), None, None, None


def linear(a, w, b, tf32: bool):
    return _Linear.apply(a, w, b, tf32)


def layer_weights(w, tf32: bool, device, rounding: str = "host"):
    """Weights the kernels multiply by: the rounded copy in TF32 mode, the fp32 values otherwise (float64)."""
    if tf32:
        w = tf32_rna_host_weights(w) if rounding == "host" else tf32_rna_device_weights(w)
    return torch.as_tensor(w).to(device=device, dtype=torch.float64)


def _maxpool_first(g: torch.Tensor, dim: int) -> torch.Tensor:
    """Max over ``dim`` whose gradient goes to the FIRST position attaining it (csrc/gather.cu)."""
    m = g.max(dim, keepdim=True).values
    k = torch.arange(g.shape[dim], device=g.device).view([-1 if i == dim else 1 for i in range(g.dim())])
    first = torch.where(g == m, k, g.shape[dim]).min(dim, keepdim=True).values
    return torch.gather(g, dim, first).squeeze(dim)


def _gather_rows(p: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """p [B,R,C], idx [B,...] -> p[b, idx[b, ...], :]."""
    B = p.shape[0]
    bsel = torch.arange(B, device=p.device).view(B, *([1] * (idx.dim() - 1)))
    return p[bsel, idx]


def read_engine_geometry(eng, t: int = 0) -> dict:
    """The resident geometry of forward slot t: per SA level l = 1..4 the level's coordinates, FPS indices and one
    ball-query index tensor per branch; per FP level f = 0..3 the 3-NN indices and interpolation weights."""
    nbr = [len(k) for k in eng._nsample]
    return {
        "xyz": {l: eng.read_geometry("xyz", l, t=t) for l in range(1, 5)},
        "fps": {l: eng.read_geometry("fps", l, t=t) for l in range(1, 5)},
        "ball": {(l, b): eng.read_geometry("ball", l, b, t=t) for l in range(1, 5) for b in range(nbr[l - 1])},
        "nn_idx": {f: eng.read_geometry("nn_idx", f, t=t) for f in range(4)},
        "nn_w": {f: eng.read_geometry("nn_w", f, t=t) for f in range(4)},
    }


def _nn_d2(fine: torch.Tensor, coarse: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    """The fp32 expansion-form squared distances the 3-NN kernels computed for the pairs ``idx`` (oracle/geom.py
    restates them bit for bit; its neighbour choice must be the engine's)."""
    from oracle import geom as G
    cidx, d2, _ = G.three_nn(fine.cpu(), coarse.cpu())
    if not torch.equal(cidx, idx.cpu().long()):
        raise AssertionError("3-NN indices differ from the C oracle's: the reference cannot restate the distances")
    return d2.to(fine.device)


def forward(desc: dict, geom: dict, x: torch.Tensor, tf32: bool, rounding: str = "host", xyz_grad: bool = False,
            control: tuple | None = None, stats: dict | None = None):
    """x [B, C, N] float64 (a leaf with requires_grad for the input gradient; its values fp32) ->
    (z [B, N, ncls] logits, l4 [B, c4, S4]) in float64, through the layers and geometry given.

    ``xyz_grad``: the walk is differentiable in the coordinates too (centres ``xyz_{l-1}[fps_idx]``, centred
    neighbour coordinates, inverse-distance weights of the squared distances ``geom["nn_d2"]`` or, without them,
    those the C oracle restates).  Every such term keeps the fp32 value the kernels used: ``v32 + (v64 - v64.detach())``.

    ``control``: a deliberately wrong reference, to show that a comparison can fail -- ("detach_skip", f): no
    gradient through the skip input of FP level f; ("swap_nn", f): 3-NN weights w0 and w1 of level f exchanged;
    ("no_xyz_w", f): no coordinate gradient through the weights of level f.

    ``stats``: filled with the fraction of active ReLUs per level ("sa1".."sa4", "fp1".."fp4", "head")."""
    dev = x.device
    ctl, ctl_f = control if control is not None else (None, -1)

    def prep(layers):
        return [(layer_weights(w, tf32, dev, rounding), torch.as_tensor(b).to(device=dev, dtype=torch.float64))
                for w, b in layers]

    def mlp(a, layers, name, relu_last=True):
        for j, (w, b) in enumerate(layers):
            a = linear(a, w, b, tf32)
            if relu_last or j + 1 < len(layers):
                a = torch.relu(a)
                if stats is not None:
                    stats.setdefault(name, []).append((a > 0).double().mean().item())
        return a

    feats = [x.permute(0, 2, 1)]                                            # [B, N, C]
    xyz = [x.detach()[:, :3].permute(0, 2, 1).float().contiguous()] + [geom["xyz"][l].float() for l in range(1, 5)]
    if xyz_grad:
        xyz64 = [x[:, :3].permute(0, 2, 1)]
        for l in range(1, 5):
            xyz64.append(_gather_rows(xyz64[l - 1], geom["fps"][l].long()))
    for l in range(1, 5):
        sa = desc["sa"][l - 1]
        outs = []
        for b in range(len(sa["radius"])):
            idx = geom["ball"][(l, b)].long()                                   # [B, S, K] into level l - 1
            rel = (_gather_rows(xyz[l - 1], idx) - xyz[l].unsqueeze(2)).to(torch.float64)   # fp32, as the kernels
            if xyz_grad:
                r64 = _gather_rows(xyz64[l - 1], idx) - xyz64[l].unsqueeze(2)
                rel = rel + (r64 - r64.detach())
            g = torch.cat([_gather_rows(feats[l - 1], idx), rel], -1)
            outs.append(_maxpool_first(mlp(g, prep(sa["mlps"][b]), f"sa{l}"), 2))
        feats.append(torch.cat(outs, -1))
    up = feats[4]
    for f in (3, 2, 1, 0):
        idx = geom["nn_idx"][f].long()
        w = geom["nn_w"][f].to(torch.float64)
        if xyz_grad and not (ctl == "no_xyz_w" and ctl_f == f):
            d2 = geom["nn_d2"][f] if "nn_d2" in geom else _nn_d2(xyz[f], xyz[f + 1], idx)
            x1, nb = xyz64[f], _gather_rows(xyz64[f + 1], idx)
            dd = -2 * (x1.unsqueeze(2) * nb).sum(-1) + (x1 ** 2).sum(-1, keepdim=True) + (nb ** 2).sum(-1)
            recip = 1.0 / (d2.to(torch.float64) + (dd - dd.detach()) + 1e-8)
            w64 = recip / recip.sum(-1, keepdim=True)
            w = w + (w64 - w64.detach())
        if ctl == "swap_nn" and ctl_f == f:
            w = w[..., [1, 0, 2]]
        interp = (_gather_rows(up, idx) * w.unsqueeze(-1)).sum(2)
        if tf32:
            interp = interp.float().to(torch.float64)
        skip = feats[f].detach() if ctl == "detach_skip" and ctl_f == f else feats[f]
        a = torch.cat([skip, interp], -1) if f > 0 else interp
        up = mlp(a, prep(desc["fp"][f]), f"fp{f + 1}")
    h = mlp(up, prep([desc["conv1"]]), "head")
    z = mlp(h, prep([desc["conv2"]]), "head", relu_last=False)
    return z, feats[4].permute(0, 2, 1)


def dz_generic(z, dlogp):
    """elementwise.cu psg_dz_from_dlogp: dz = dlogp - softmax * sum(dlogp)."""
    return dlogp - torch.softmax(z, -1) * dlogp.sum(-1, keepdim=True)


def dz_ce(z, labels, scale):
    """psg_dz_ce: (softmax - onehot) * scale."""
    p = torch.softmax(z, -1)
    return (p - torch.nn.functional.one_hot(labels.long(), z.shape[-1]).to(p.dtype)) * scale


def dz_cw(z, labels, sgn, kappa):
    """psg_dz_cw (psg_loss.cuh): f = clamp(sgn (p_y - max_{c != y} p_c), min = -kappa); dz = p (g - <g, p>) with
    g = df/dp, the competing class the first maximum among c != y."""
    p = torch.softmax(z, -1)
    y = labels.long().unsqueeze(-1)
    onehot = torch.zeros_like(p).scatter_(-1, y, 1.0)
    other = torch.where(onehot > 0, torch.zeros_like(p), p)
    oc = other.argmax(-1, keepdim=True)                                       # first maximum
    py, po = p.gather(-1, y), p.gather(-1, oc)
    passed = (sgn * (py - po) >= -kappa).to(p.dtype)
    g = onehot * (sgn * passed) - torch.zeros_like(p).scatter_(-1, oc, 1.0) * (sgn * passed)
    dot = (g * p).sum(-1, keepdim=True)
    return p * (g - dot)


def input_gradient(z, x, dz, retain_graph: bool = True):
    """d x of <z, dz> through the feature path: [B, C, N]."""
    (g,) = torch.autograd.grad(z, x, dz, retain_graph=retain_graph)
    return g


# ------------------------------------------------------------------------------------------------
# the engine against the walk above: one harness for every GPU test that compares whole networks
# ------------------------------------------------------------------------------------------------
KAPPA = 0.2


def prof_counts() -> dict:
    """Launch counts per family since the last call (psg_prof)."""
    import ctypes as C
    from pointsecguard_b200 import _lib as L
    n = L.psg_prof_ncat()
    ms, cnt = (C.c_double * n)(), (C.c_int64 * n)()
    assert L.psg_prof_collect(ms, cnt) == 0
    return {L.psg_prof_name(i).decode(): int(cnt[i]) for i in range(n)}


def grad_stats(mine, ref):
    """(relative Frobenius error, sign agreement on the nonzero reference elements, fraction within rtol 1e-3)."""
    mine, ref = mine.double(), ref.double()
    rel = ((mine - ref).norm() / ref.norm()).item()
    nz = ref != 0
    sign = (torch.sign(mine[nz]) == torch.sign(ref[nz])).double().mean().item()
    close = ((mine - ref).abs() <= 1e-3 * ref.abs() + 1e-12).double().mean().item()
    return rel, sign, close


def engine_inputs(B: int, N: int, kind: str = "uniform", in_channels: int = 9, num_classes: int = 13, seed: int = 0):
    """Synthetic blocks (channels 0:3 coordinates; channels past the nine of synthetic.make_blocks uniform in [0, 1)),
    z-band labels folded into the class range, and a random d logp; on cuda."""
    from pointsecguard_b200 import synthetic as syn
    x = syn.make_blocks(B, N, seed, kind)
    lab = (syn.zband_labels(x) % num_classes).to(torch.int32).view(-1)
    if in_channels <= 9:
        x = x[:, :in_channels]
    else:
        extra = torch.rand(B, in_channels - 9, N, generator=torch.Generator().manual_seed(seed + 2))
        x = torch.cat([x, extra], 1)
    dlogp = torch.randn(B, N, num_classes, generator=torch.Generator().manual_seed(seed + 1)) / N
    return x.contiguous().cuda(), lab.cuda(), dlogp.cuda()


def run_engine(desc: dict, inputs, mode: int, sa_compact: int = 1, xyz_grad: bool = False):
    """Forward, the three loss kinds and the backward on a fresh engine; each loss once after forward(want_logp=True)
    and once after forward(want_logp=False) (the deferred fp1 + head pass).  Returns the outputs, the launch counts of
    the first forward + backward and the geometry."""
    from pointsecguard_b200 import _lib as L
    from pointsecguard_b200.engine import Engine
    x, lab, dlogp = inputs
    B, _, N = x.shape
    eng = Engine(desc, torch.device("cuda", 0), mode)
    out = {}
    L.psg_set_option(b"sa_compact", sa_compact)
    try:
        eng.bind(B, N, 1)
        eng.set_input(x)
        eng.set_xyz_grad(xyz_grad)
        torch.manual_seed(0)
        eng.geometry(eng.draw_starts(1))
        losses = {0: lambda: eng.loss_grad_generic(dlogp), 1: lambda: eng.loss_grad_ce(lab, -1, 1.0 / N),
                  2: lambda: eng.loss_grad_cw(lab, -1, 1.0, KAPPA)}
        prof_counts()
        L.psg_prof_enable(1)
        try:
            out["logp"], out["l4"] = eng.forward(0, True, True)
            losses[0]()
            out[(0, True)] = eng.backward(0)
            counts = prof_counts()
        finally:
            L.psg_prof_enable(0)
        for k in (1, 2):
            eng.forward(0, True, False)
            losses[k]()
            out[(k, True)] = eng.backward(0)
        for k in (0, 1, 2):
            eng.forward(0, False, False)
            losses[k]()
            out[(k, False)] = eng.backward(0)
        geom = read_engine_geometry(eng)
        torch.cuda.synchronize()
    finally:
        L.psg_set_option(b"sa_compact", 1)
    return out, counts, geom


def reference(desc: dict, geom: dict, inputs, tf32: bool, xyz_grad: bool = False, control=None, stats=None):
    """Log-probabilities, l4 and the input gradient of each loss kind through the walk above (float64)."""
    x0, lab, dlogp = inputs
    B, _, N = x0.shape
    x = x0.double().requires_grad_(True)
    z, l4 = forward(desc, geom, x, tf32, xyz_grad=xyz_grad, control=control, stats=stats)
    lab2 = lab.view(B, N)
    dz = {0: dz_generic(z, dlogp.double()), 1: dz_ce(z, lab2, 1.0 / N), 2: dz_cw(z, lab2, 1.0, KAPPA)}
    res = {"logp": torch.log_softmax(z, -1).detach(), "l4": l4.detach()}
    for k in (0, 1, 2):
        res[k] = input_gradient(z, x, dz[k].detach(), retain_graph=k < 2)
    return res


def compare(out: dict, ref: dict, tag: str, what: str, channels=slice(None)):
    """Worst deviations of the engine's outputs from a reference: (logp max |d|, l4 max |d| / max |l4|,
    (grad rel, sign, within-rtol-1e-3) worst over the six gradients, on ``channels``).  Prints them."""
    lp = (out["logp"].double() - ref["logp"]).abs().max().item()
    l4 = ((out["l4"].double() - ref["l4"]).abs().max() / ref["l4"].abs().max()).item()
    grads = {key: grad_stats(out[key][:, channels], ref[key[0]][:, channels]) for key in out if isinstance(key, tuple)}
    worst = (max(g[0] for g in grads.values()), min(g[1] for g in grads.values()), min(g[2] for g in grads.values()))
    print(f"{tag} vs {what}: logp {lp:.2e} l4 {l4:.2e} grad rel {worst[0]:.2e} sign {worst[1]:.6f} "
          f"within-rtol-1e-3 {worst[2]:.5f}")
    for key, g in sorted(grads.items()):
        print(f"    loss kind {key[0]} want_logp={key[1]}: rel {g[0]:.2e} sign {g[1]:.6f} close {g[2]:.5f}")
    return lp, l4, worst
