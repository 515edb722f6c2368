"""The tcgen05 TF32 network (engine.MLP_TF32: fused set-abstraction kernels, streamed SA3 / SA4, FP tile programs,
the fp1 + head chain) against the TF32-exact reference of oracle/tf32_oracle.py, at the batch sizes that select each
fused path, on the trained checkpoint.

The reference applies the two roundings the hardware applies -- weights rounded to nearest TF32 after the truncation
compensation, operands truncated to 19 bits in front of every product -- inside an fp64 computation, and reads the
geometry the engine computed.  One layer of it matches the kernels to 1e-6 of the output scale (test_gpu_gemm.py).
Through the whole network it cannot be as close: truncation is discontinuous, so an fp32 summation-order difference
of one ulp flips the truncated operand by a whole TF32 ulp whenever it straddles a truncation boundary, and those
flips compound layer after layer.  On the trained checkpoint, which amplifies input noise by ~300x (the fp32 mode
against the plain fp64 reference below: logp 2e-5 from fp32 rounding alone), the kernels then sit about a sixth as
far from the TF32-exact reference as from the unrounded one.  The gates below hold that: every fused path at every
batch size must stay within them and well closer to the TF32-exact reference than to the plain one -- a tail tile or
row block computed wrong, a dropped ReLU mask, or a path without the compensation lands at the plain distance or
beyond.  Every test prints both deviations.

Measured on a B200 (1000 W), worst case over the 12 cases:
                          vs TF32-exact   vs plain fp64 (best case)   gate
    logp max |d|          1.5e-2          7.6e-2                      3e-2
    l4 max |d| / max|l4|  1.4e-3          5.6e-3                      3e-3
    grad rel (Frobenius)  5.4e-2          1.3e-1                      8e-2
    sign agreement        0.9850          0.959                       0.975
and per case the plain deviation is at least 2.8x (gradient) and 4.5x (logp) the TF32-exact one (asserted: 2x).
"""
import numpy as np
import pytest
import torch

from oracle import tf32_oracle as TO
from pointsecguard_b200 import synthetic as syn

LOGP_GATE = 3e-2
L4_GATE = 3e-3
GRAD_REL_GATE = 8e-2
SIGN_GATE = 0.975
SHARP = 2.0               # the plain reference must sit at least this many times farther than the TF32-exact one

# fp32-grade modes against the plain fp64 reference on the trained checkpoint (measured on a B200: fp32 logp <= 2.9e-5,
# grad rel <= 2.4e-3, sign >= 0.99985; 3xTF32 logp <= 1.8e-4, grad rel <= 3.5e-3, sign >= 0.99958).  The gradient gates
# are looser than tests/test_gpu_model.py's (rel 1e-4 on the default-init network): on the trained checkpoint a max-pool
# arg-max that flips under fp32 rounding at SA3 / SA4 re-routes the gradient of a sixteenth of the block.
FP32_LOGP_ATOL = 1e-3
FP32_GRAD_REL, FP32_SIGN = 1e-2, 0.999

N = 4096


# ------------------------------------------------------------------------------------------------
# CPU: the reference itself
# ------------------------------------------------------------------------------------------------
def _tf32_rna_c(a: np.ndarray) -> np.ndarray:
    """csrc/net.cu tf32_rna restated on uint32 bit patterns (numpy)."""
    with np.errstate(over="ignore"):
        u = np.asarray(a, dtype=np.float64).astype(np.float32).view(np.uint32).astype(np.uint64)
    r = np.where((u & 0x7F800000) != 0x7F800000, (u + 0x1000) & 0xFFFFE000, u)
    return r.astype(np.uint32).view(np.float32)


def test_tf32_rounding_is_bit_identical_to_the_library():
    f32 = np.float32
    edge = np.array([0.0, -0.0, 1.0, -1.0, 1.0 + 2.0 ** -11, 1.0 + 2.0 ** -10 + 2.0 ** -11, 1.0 - 2.0 ** -12,
                     float(np.finfo(f32).max), -float(np.finfo(f32).max), float(np.finfo(f32).tiny), 1e-45,
                     2.0 ** 128 * 0.99999999, np.inf, -np.inf, np.nan, 3.4028235e38, 0.1, -0.3, 65504.0])
    rnd = np.random.default_rng(0).standard_normal(200000) * np.exp(np.random.default_rng(1).uniform(-40, 40, 200000))
    for v in (edge, rnd):
        got = TO.tf32_rna(torch.from_numpy(v)).numpy()
        want = _tf32_rna_c(v)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # ties round away from zero in magnitude; the carry may move into the exponent
    assert TO.tf32_rna(torch.tensor([1.0 + 2.0 ** -11])).item() == 1.0 + 2.0 ** -10
    assert TO.tf32_rna(torch.tensor([2.0 - 2.0 ** -12])).item() == 2.0
    # truncation keeps the top 19 bits
    t = TO.tf32_trunc(torch.from_numpy(rnd)).numpy().view(np.uint32)
    assert np.array_equal(t, rnd.astype(np.float32).view(np.uint32) & np.uint32(0xFFFFE000))
    # the device rounding multiplies in fp32 by 1.f + 3.45e-4f
    w = np.random.default_rng(2).standard_normal(4096).astype(np.float32)
    dev = TO.tf32_rna_device_weights(torch.from_numpy(w)).numpy()
    want = _tf32_rna_c((w * (np.float32(1.0) + np.float32(3.45e-4))).astype(np.float32))
    assert np.array_equal(dev.view(np.uint32), want.view(np.uint32))
    host = TO.tf32_rna_host_weights(torch.from_numpy(w)).numpy()
    assert np.array_equal(host.view(np.uint32), _tf32_rna_c(w.astype(np.float64) * (1.0 + 3.45e-4)).view(np.uint32))


def _cpu_geometry(x, arch):
    """Geometry of one forward from the C oracle, drawing the FPS starts on the global generator in the reference's
    order (as OracleModel does)."""
    from oracle import geom as G
    from oracle import pointnet2_oracle as PO
    B = x.shape[0]
    xyz = [x[:, :3].permute(0, 2, 1).contiguous()]
    geom = {"xyz": {}, "fps": {}, "ball": {}, "nn_idx": {}, "nn_w": {}, "nn_d2": {}}
    for l, (S, radii, ks) in enumerate(PO._SA[arch], start=1):
        start = torch.randint(0, xyz[-1].shape[1], (B,), dtype=torch.long)
        fps = G.fps(xyz[-1], S, start)
        new = PO.index_points(xyz[-1], fps)
        for b, (r, K) in enumerate(zip(radii, ks)):
            geom["ball"][(l, b)] = G.ball_query(r, K, xyz[-1], new)
        geom["xyz"][l], geom["fps"][l] = new, fps
        xyz.append(new)
    for f in range(4):
        idx, d2, w = G.three_nn(xyz[f], xyz[f + 1])
        geom["nn_idx"][f], geom["nn_w"][f], geom["nn_d2"][f] = idx, w, d2
    return geom


@pytest.mark.parametrize("arch", ["ssg", "msg"])
def test_plain_reference_matches_the_cpu_oracle(arch):
    """The network walk of tf32_oracle (plain fp64 mode, differentiable in the coordinates) against the CPU oracle
    model (unfolded BatchNorm, its own geometry, autograd through centres, centred neighbours and inverse-distance
    weights) at B = 1, N = 1024: log-probabilities and the input gradient on all nine channels.  The TF32 mode of the
    same walk differs from both by the TF32 rounding and no more."""
    from oracle import pointnet2_oracle as PO
    if arch == "ssg":
        from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    else:
        from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_model
    sd = syn.load_checkpoint(arch)
    m = get_model(13)
    m.load_state_dict(sd)
    desc = m.eval().describe()
    x0 = syn.make_blocks(1, 1024, 0, "uniform")
    y = syn.zband_labels(x0).long()
    torch.manual_seed(0)
    geom = _cpu_geometry(x0, arch)
    xo = x0.double().requires_grad_(True)
    torch.manual_seed(0)
    lo, _ = PO.OracleModel({k: v.double() if v.is_floating_point() else v for k, v in sd.items()}, arch)(xo)
    (torch.nn.functional.nll_loss(lo.reshape(-1, 13), y.view(-1), reduction="sum") / 1024).backward()
    res = {}
    for tf32 in (False, True):
        x = x0.double().requires_grad_(True)
        z, l4 = TO.forward(desc, geom, x, tf32, xyz_grad=True)
        g = TO.input_gradient(z, x, TO.dz_ce(z, y.view(1, -1), 1.0 / 1024))
        res[tf32] = (torch.log_softmax(z, -1).detach(), g)
    go = xo.grad
    lp, g = res[False]
    err = (lp - lo.detach()).abs().max().item()
    rel = ((g - go).norm() / go.norm()).item()
    rel_xyz = ((g[:, :3] - go[:, :3]).norm() / go[:, :3].norm()).item()
    lp1, g1 = res[True]
    err1 = (lp1 - lo.detach()).abs().max().item()
    rel1 = ((g1 - go).norm() / go.norm()).item()
    # without the coordinate terms channels 0:3 carry the feature path only, far from the oracle's
    x = x0.double().requires_grad_(True)
    z, _ = TO.forward(desc, geom, x, False)
    gf = TO.input_gradient(z, x, TO.dz_ce(z, y.view(1, -1), 1.0 / 1024))
    rel_f = ((gf[:, :3] - go[:, :3]).norm() / go[:, :3].norm()).item()
    print(f"{arch}: plain vs oracle logp {err:.2e} grad rel {rel:.2e} (xyz {rel_xyz:.2e}, features-only walk "
          f"{rel_f:.2e}) | tf32 vs oracle logp {err1:.2e} grad rel {rel1:.2e}")
    # what is left is the BatchNorm folding, whose weights describe() stores in fp32
    assert err < 1e-4 and rel < 1e-4 and rel_xyz < 1e-4
    assert rel_f > 1e-2
    assert 1e-3 < err1 < 0.5 and 1e-3 < rel1 < 0.5


# ------------------------------------------------------------------------------------------------
# GPU: the engine against the reference
# ------------------------------------------------------------------------------------------------
_MODELS = {}


def _model(arch):
    if arch not in _MODELS:
        if arch == "ssg":
            from pointsecguard_b200.models.pointnet2_sem_seg import get_model
        else:
            from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_model
        m = get_model(13)
        m.load_state_dict(syn.load_checkpoint(arch))
        _MODELS[arch] = m.eval()
    return _MODELS[arch]


def _run_engine(arch, B, kind, mode, sa_compact=1):
    desc = _model(arch).describe()
    inputs = TO.engine_inputs(B, N, kind)
    out, counts, geom = TO.run_engine(desc, inputs, mode, sa_compact)
    return out, counts, geom, desc, inputs


def _compare(out, ref, arch, B, what):
    return TO.compare(out, ref, f"{arch} B={B}", what)


# (arch, B, cloud kind, sa_compact): fp2 (B * 1024 rows) is a tile program from 48 row tiles on, i.e. B >= 6, fp3
# (B * 256 rows) from B >= 24 (SSG only: MSG's fp3 input is wider than the operand buffer, as is fp4's everywhere)
CASES = [
    ("ssg", 2, "uniform", 1), ("ssg", 2, "duplicates", 1), ("ssg", 5, "uniform", 1), ("ssg", 6, "uniform", 1),
    ("ssg", 16, "uniform", 1), ("ssg", 16, "clustered", 1), ("ssg", 24, "uniform", 1), ("ssg", 6, "uniform", 0),
    ("msg", 8, "uniform", 1), ("msg", 8, "duplicates", 1), ("msg", 24, "uniform", 1), ("msg", 24, "duplicates", 1),
]


def _expected_counts(arch, B):
    """Launches of one forward(want_logp=True) + backward in the TF32 mode.  SSG: all four SA levels fused (SA1, SA2)
    or streamed (SA3, SA4); MSG: SA1 - SA3 both branches, SA4 (1024-wide input) per layer."""
    sa = 4 if arch == "ssg" else 6
    fp = (B * 1024 // 128 >= 48) + (arch == "ssg" and B * 256 // 128 >= 48)
    return {"sa_fused_fwd": sa, "sa_fused_bwd": sa, "fp_fused_fwd": fp, "fp_fused_bwd": fp, "head_chain": 2}


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[f"{a}-B{b}-{k}" + ("" if c else "-padded") for a, b, k, c in CASES])
def test_tf32_network_vs_tf32_exact_reference(case):
    from pointsecguard_b200.engine import MLP_TF32
    arch, B, kind, compact = case
    out, counts, geom, desc, inputs = _run_engine(arch, B, kind, MLP_TF32, compact)
    want = _expected_counts(arch, B)
    got = {k: counts[k] for k in want}
    print(f"{arch} B={B} {kind} compact={compact}: launches {got}")
    assert got == want
    exact = TO.reference(desc, geom, inputs, tf32=True)
    lp, l4, (rel, sign, _) = _compare(out, exact, arch, B, "TF32-exact")
    plain = TO.reference(desc, geom, inputs, tf32=False)
    lp0, _, (rel0, _, _) = _compare(out, plain, arch, B, "plain fp64")
    assert lp < LOGP_GATE and l4 < L4_GATE
    assert rel < GRAD_REL_GATE and sign >= SIGN_GATE
    # the kernels follow the rounded arithmetic, not merely the unrounded one
    assert lp0 >= SHARP * lp and rel0 >= SHARP * rel


CONTROL = [(0, "ssg", 2, "uniform"), (0, "ssg", 16, "uniform"), (0, "msg", 8, "uniform"),
           (2, "ssg", 6, "uniform"), (2, "ssg", 16, "uniform"), (2, "ssg", 24, "uniform")]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CONTROL, ids=[f"{'fp32' if m == 0 else 'x3'}-{a}-B{b}" for m, a, b, _ in CONTROL])
def test_fp32_grade_modes_vs_plain_reference(case):
    """The fp32 mode (a control of the harness: if it fails the harness is wrong, not the kernels) and the 3xTF32 mode
    against the plain fp64 reference through the same walk (gates: FP32_* above)."""
    mode, arch, B, kind = case
    out, _, geom, desc, inputs = _run_engine(arch, B, kind, mode)
    plain = TO.reference(desc, geom, inputs, tf32=False)
    lp, l4, (rel, sign, _) = _compare(out, plain, arch, B, f"plain fp64 (mode {mode})")
    assert lp < FP32_LOGP_ATOL and l4 < 1e-4
    assert rel < FP32_GRAD_REL and sign >= FP32_SIGN


@pytest.mark.gpu
def test_one_nb_step_follows_the_tf32_exact_gradient_at_bench_size():
    """One NB_attack step on the TF32 model at B = 16: the colour moves by alpha * sign of the CE gradient, so
    sign(adv - x) on channels 3:6 must follow the sign of the TF32-exact gradient of the geometry that step used more
    closely than that of the plain gradient.  Elements with |g| < 1e-6 max|g| are left out (their sign is rounding
    noise).  Measured on a B200: 0.9894 against the TF32-exact gradient, 0.9552 against the plain one."""
    from pointsecguard_b200 import torchattacks
    from pointsecguard_b200.engine import MLP_FP32, MLP_TF32
    m = _model("ssg").cuda()
    m.set_mlp_mode(MLP_TF32)
    try:
        B = 16
        x = syn.make_blocks(B, N, 0, "uniform").cuda()
        lab = syn.zband_labels(x.cpu())
        torch.manual_seed(0)
        adv = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=1)(x, lab.numpy().astype(np.float64))
        geom = TO.read_engine_geometry(m.engine(x.device))
        desc = m.describe()
    finally:
        m.set_mlp_mode(MLP_FP32)
    step = torch.sign(adv[:, 3:6] - x[:, 3:6]).double()
    agree = {}
    for tf32 in (True, False):
        xr = x.double().requires_grad_(True)
        z, _ = TO.forward(desc, geom, xr, tf32)
        g = TO.input_gradient(z, xr, TO.dz_ce(z, lab.cuda().view(B, N), 1.0 / N), retain_graph=False)[:, 3:6]
        keep = g.abs() >= 1e-6 * g.abs().max()
        agree[tf32] = (step[keep] == torch.sign(g[keep])).double().mean().item()
    print(f"NB step sign agreement: TF32-exact {agree[True]:.6f}, plain fp64 {agree[False]:.6f}")
    assert agree[True] >= SIGN_GATE and agree[True] > agree[False]
