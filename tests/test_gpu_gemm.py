"""The shared-MLP GEMM kernels through the C ABI (psg_mlp_forward / psg_mlp_backward) against fp64 torch references:
fp32 CUDA-core kernel (mode 0) and error-compensated 3xTF32 tcgen05 kernel (mode 2) against the plain product at
rtol 1e-5 of the output scale; tcgen05 TF32 kernel (mode 1) against the TF32-exact layer of oracle/tf32_oracle.py
(weights rounded like the library rounds them, operands truncated to 19 bits like the tensor core reads them), which
leaves only the fp32 accumulation to tolerate.

Measured on a B200 over the cases below (max error / output scale): fp32 <= 8.1e-7, 3xTF32 <= 2.4e-6; TF32 against
the TF32-exact layer <= 2.1e-6 (host-rounded weights), against the plain product >= 1.6e-4 -- so the gate TF32_EXACT_TOL
is five times the first and a fifteenth of the second: a layer fed the uncompensated weight copy, or whose operands
were rounded instead of truncated, misses it."""
import numpy as np
import pytest
import torch

from oracle import tf32_oracle as TO

pytestmark = pytest.mark.gpu

CASES = [  # rows, cin (k1, k2), cout
    (256, (16, 0), 32), (1000, (80, 0), 64), (128, (272, 0), 256), (4096, (128, 0), 128),
    (300, (256, 512), 256), (512, (208, 0), 256), (640, (128, 0), 13), (128, (64, 64), 96), (384, (512, 0), 208),
    # single rows and the edges of one 128-row tile; 80 + 48 columns = 20 + 12 planes: a whole number of 16-plane weight
    # boxes in all, but each source ends in a short stage (the tensor-map weight load once hung there)
    (1, (64, 0), 64), (127, (128, 0), 96), (129, (80, 48), 128),
    # more CTAs than SMs (gemm_tc.cu kBigCtas): 150 tiles of K = 64 (mode 1: 16 KB stages; mode 2: bn 64, one-stage
    # ring), 157 x 1 tiles of K = 512 and 513 tiles of K = 128 (mode 1: 8-plane stages; mode 2: bn 64, one stage);
    # the dgrad of each runs with the roles of K and the output width swapped
    (19200, (64, 0), 64), (20000, (512, 0), 128), (65541, (128, 0), 128),
]
TF32_EXACT_TOL = 1e-5
PLAIN_TOL = 1e-5


def _mk(rows, k1, k2, cout, seed):
    g = torch.Generator().manual_seed(seed)
    a1 = torch.randn(rows, k1, generator=g).cuda()
    a2 = torch.randn(rows, k2, generator=g).cuda() if k2 else None
    w = (torch.randn(cout, k1 + k2, generator=g) / np.sqrt(k1 + k2)).contiguous()
    b = torch.randn(cout, generator=g).contiguous()
    return a1, a2, w, b


def _run_layer(m, a1, a2, rows, cout, mode):
    """Forward with ReLU, then the dgrad of a random upstream gradient under the ReLU mask of a lower layer."""
    from pointsecguard_b200 import _lib as L
    from pointsecguard_b200.tlayout import TTensor
    st = torch.cuda.current_stream().cuda_stream
    k2 = a2.shape[1] if a2 is not None else 0
    t1 = TTensor.from_rowmajor(a1)
    t2 = TTensor.from_rowmajor(a2) if k2 else None
    out = TTensor(rows, cout, "cuda")
    assert L.psg_mlp_forward(m, t1.ptr, t1.wchunks, 0, t1.wchunks, t2.ptr if k2 else None, t2.wchunks if k2 else 0, 0,
                             t2.wchunks if k2 else 0, rows, out.ptr, out.wchunks, 1, mode, st) == 0
    y = out.to_rowmajor()
    g = torch.Generator(device="cuda").manual_seed(rows + cout)
    dy = TTensor.from_rowmajor(torch.randn(rows, cout, device="cuda", generator=g))
    kp = t1.cpad + (t2.cpad if k2 else 0)
    maskt = TTensor.from_rowmajor(torch.randn(rows, kp, device="cuda", generator=g))
    dx = TTensor(rows, kp, "cuda")
    assert L.psg_mlp_backward(m, dy.ptr, dy.wchunks, rows, dx.ptr, dx.wchunks, maskt.ptr, maskt.wchunks, mode, st) == 0
    return y, dx.to_rowmajor(), dy.to_rowmajor(), maskt.to_rowmajor(), t1.cpad


def _reference(a1, a2, w, b, dyr, mk, cpad1, tf32, rounding="host"):
    """fp64 forward and masked dgrad, with the TF32 roundings of the tensor core (tf32=True) or without."""
    k1 = a1.shape[1]
    k2 = a2.shape[1] if a2 is not None else 0
    a = torch.cat([a1, a2], 1) if k2 else a1
    wd = TO.layer_weights(w, tf32, "cuda", rounding)
    bd = b.cuda().double()
    ad = TO.tf32_trunc(a).double() if tf32 else a.double()
    ref = torch.relu(ad @ wd.t() + bd)
    dd = TO.tf32_trunc(dyr).double() if tf32 else dyr.double()
    refdx = dd @ wd
    rows = a.shape[0]
    if k2:   # padded two-source layout: [k1 | pad | k2 | pad]
        full = torch.zeros(rows, mk.shape[1], dtype=torch.float64, device="cuda")
        full[:, :k1] = refdx[:, :k1]
        full[:, cpad1: cpad1 + k2] = refdx[:, k1:]
        refdx = full
    else:
        mk = mk[:, : k1]
    return ref, refdx * (mk > 0)


def _rel_err(got, ref):
    return (got.double() - ref).abs().max().item() / ref.abs().max().item()


@pytest.mark.parametrize("mode", [0, 1, 2], ids=["fp32", "tf32", "x3"])
@pytest.mark.parametrize("case", CASES, ids=[f"{c[0]}x{c[1][0]}+{c[1][1]}->{c[2]}" for c in CASES])
def test_mlp_forward_backward(case, mode):
    from pointsecguard_b200 import _lib as L
    rows, (k1, k2), cout = case
    a1, a2, w, b = _mk(rows, k1, k2, cout, rows + cout)
    m = L.psg_mlp_create(w.data_ptr(), b.data_ptr(), k1 + k2, cout)
    assert m
    try:
        y, dx, dyr, mk, cpad1 = _run_layer(m, a1, a2, rows, cout, mode)
    finally:
        L.psg_mlp_destroy(m)
    got_dx = dx if k2 else dx[:, : k1]
    plain = _reference(a1, a2, w, b, dyr, mk, cpad1, tf32=False)
    e_plain = (_rel_err(y, plain[0]), _rel_err(got_dx, plain[1]))
    if mode == 1:
        exact = _reference(a1, a2, w, b, dyr, mk, cpad1, tf32=True)
        e = (_rel_err(y, exact[0]), _rel_err(got_dx, exact[1]))
        print(f"tf32 {case}: fwd {e[0]:.2e} dgrad {e[1]:.2e} of scale (vs the plain product {e_plain[0]:.2e} {e_plain[1]:.2e})")
        assert e[0] <= TF32_EXACT_TOL and e[1] <= TF32_EXACT_TOL
        # the gate is sharp: an unrounded weight copy or untruncated operands would miss it
        assert min(e_plain) >= 10 * TF32_EXACT_TOL
    else:
        print(f"mode {mode} {case}: fwd {e_plain[0]:.2e} dgrad {e_plain[1]:.2e} of scale")
        assert e_plain[0] <= PLAIN_TOL and e_plain[1] <= PLAIN_TOL


DEVICE_CASES = [(256, (16, 0), 32), (300, (256, 512), 256), (129, (80, 48), 128), (20000, (512, 0), 128)]


@pytest.mark.parametrize("case", DEVICE_CASES, ids=[f"{c[0]}x{c[1][0]}+{c[1][1]}->{c[2]}" for c in DEVICE_CASES])
def test_device_loaded_layer(case):
    """Layers whose weights live in device memory (psg_mlp_create_device + psg_mlp_load, the trainer's layers): packed
    on the device by repack_kernel.  Mode 0 is bit-identical to a host-built layer of the same weights; mode 1 matches
    the TF32-exact layer with the device's rounding (product with 1 + 3.45e-4 taken in fp32)."""
    from pointsecguard_b200 import _lib as L
    rows, (k1, k2), cout = case
    a1, a2, w, b = _mk(rows, k1, k2, cout, rows + cout + 1)
    wd, bd = w.cuda(), b.cuda()
    host = L.psg_mlp_create(w.data_ptr(), b.data_ptr(), k1 + k2, cout)
    dev = L.psg_mlp_create_device(k1 + k2, cout)
    assert host and dev
    try:
        assert L.psg_mlp_load(dev, wd.data_ptr(), bd.data_ptr(), torch.cuda.current_stream().cuda_stream) == 0
        r_host = _run_layer(host, a1, a2, rows, cout, 0)
        r_dev = _run_layer(dev, a1, a2, rows, cout, 0)
        assert torch.equal(r_host[0], r_dev[0]) and torch.equal(r_host[1], r_dev[1])
        y, dx, dyr, mk, cpad1 = _run_layer(dev, a1, a2, rows, cout, 1)
    finally:
        L.psg_mlp_destroy(host)
        L.psg_mlp_destroy(dev)
    got_dx = dx if k2 else dx[:, : k1]
    exact = _reference(a1, a2, w, b, dyr, mk, cpad1, tf32=True, rounding="device")
    e = (_rel_err(y, exact[0]), _rel_err(got_dx, exact[1]))
    plain = _reference(a1, a2, w, b, dyr, mk, cpad1, tf32=False)
    e_plain = (_rel_err(y, plain[0]), _rel_err(got_dx, plain[1]))
    print(f"device-loaded tf32 {case}: fwd {e[0]:.2e} dgrad {e[1]:.2e} (vs the plain product {e_plain[0]:.2e} {e_plain[1]:.2e})")
    assert e[0] <= TF32_EXACT_TOL and e[1] <= TF32_EXACT_TOL
    assert min(e_plain) >= 10 * TF32_EXACT_TOL


def test_model_tf32_mode_close_to_fp32():
    """Whole network with tcgen05 TF32 MLPs: same geometry (bit-exact indices), log-probabilities
    within 5e-3 absolute of the fp32 path, identical predictions on > 99.5 % of the points."""
    from pointsecguard_b200 import synthetic as syn
    from pointsecguard_b200.engine import MLP_FP32, MLP_TF32
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    m = get_model(13)
    m.load_state_dict(syn.make_state_dict("ssg"))
    m = m.cuda().eval()
    x = syn.make_blocks(2, 4096, 0).cuda()
    torch.manual_seed(0)
    ref, _ = m(x)
    m.set_mlp_mode(MLP_TF32)
    torch.manual_seed(0)
    out, _ = m(x)
    m.set_mlp_mode(MLP_FP32)
    err = (out - ref).abs().max().item()
    agree = (out.argmax(2) == ref.argmax(2)).float().mean().item()
    print("tf32 vs fp32: max |dlogp|", err, "argmax agreement", agree)
    assert err < 5e-3 and agree > 0.995


@pytest.mark.parametrize("arch", ["ssg", "msg"])
def test_model_tf32_gradient_close_to_fp32(arch):
    """tcgen05 mode (fused set-abstraction kernels, TF32 MLPs) against the fp32 parity mode: same
    indices, log-probabilities within 5e-3, input gradient within 8e-2 relative (Frobenius) with
    > 99 % sign agreement -- the stated, looser TF32 tolerance (SURVEY.md App. B: 2^-11 weight noise
    alone gives 4e-2 / 99.7 %)."""
    from pointsecguard_b200 import synthetic as syn
    from pointsecguard_b200.engine import MLP_FP32, MLP_TF32
    if arch == "ssg":
        from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    else:
        from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_model
    m = get_model(13)
    m.load_state_dict(syn.make_state_dict(arch))
    m = m.cuda().eval()
    x0 = syn.make_blocks(2, 4096, 0).cuda()
    res = {}
    for mode in (MLP_FP32, MLP_TF32):
        m.set_mlp_mode(mode)
        x = x0.clone().requires_grad_(True)
        torch.manual_seed(0)
        logp, l4 = m(x)
        y = (logp.detach().argmax(2) + 1) % 13 if mode == MLP_FP32 else res["y"]
        res["y"] = y
        cost = torch.nn.functional.cross_entropy(logp.reshape(-1, 13), y.view(-1), reduction="sum") / logp.size(1)
        cost.backward()
        res[mode] = (logp.detach(), l4, x.grad[:, 3:].clone())
    m.set_mlp_mode(MLP_FP32)
    (lp0, l40, g0), (lp1, l41, g1) = res[MLP_FP32], res[MLP_TF32]
    err = (lp1 - lp0).abs().max().item()
    l4err = ((l41 - l40).abs().max() / l40.abs().max()).item()
    rel = ((g1 - g0).norm() / g0.norm()).item()
    nz = g0 != 0
    sign = (torch.sign(g1[nz]) == torch.sign(g0[nz])).float().mean().item()
    zero_same = ((g1 == 0) == (g0 == 0)).float().mean().item()
    print(f"{arch}: tf32 vs fp32 |dlogp| {err:.2e} l4 rel {l4err:.2e} grad rel {rel:.2e} sign {sign:.5f} zero-pattern {zero_same:.5f}")
    assert err < 5e-3 and l4err < 5e-3 and rel < 8e-2 and sign > 0.99 and zero_same > 0.999


def test_attack_metrics_tf32_vs_fp32_within_half_a_point():
    """north_star gate: accuracy / mIoU / attack success after the attack agree within +-0.5 pt between
    the tcgen05 TF32 path and the fp32 parity path (same seeds, bit-identical geometry)."""
    from pointsecguard_b200 import metrics as MT, synthetic as syn, torchattacks
    from pointsecguard_b200.engine import MLP_FP32, MLP_TF32
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    m = get_model(13)
    m.load_state_dict(syn.make_state_dict("ssg", init="he"))  # input-sensitive random network (synthetic.py)
    m = m.cuda().eval()
    x = syn.make_blocks(16, 4096, 3).cuda()                   # 65536 points: the gate is on aggregate metrics
    torch.manual_seed(5)
    lab = m(x)[0].argmax(2)                                  # clean predictions: initial accuracy 100 %
    zl = syn.zband_labels(x.cpu())
    mask = zl == 11
    res = {}
    for mode in (MLP_FP32, MLP_TF32):
        m.set_mlp_mode(mode)
        torch.manual_seed(0)
        adv = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=10)(x, lab.cpu().numpy().astype(np.float64))
        torch.manual_seed(1)
        s1 = MT.summarize(MT.attack_counters(m(adv)[0], lab))
        torch.manual_seed(0)
        advt = torchattacks.tar_NB_attack(m, eps=0.5, alpha=0.1, iters=10, target=7, mask=mask)(x, zl.numpy().astype(np.float64))
        torch.manual_seed(1)
        s2 = MT.summarize(MT.attack_counters(m(advt)[0], zl.cuda(), mask.cuda(), 7))
        res[mode] = (s1, s2, adv)
    m.set_mlp_mode(MLP_FP32)
    (a1, a2, adv0), (b1, b2, adv1) = res[MLP_FP32], res[MLP_TF32]
    print("NB  fp32", a1, "\n    tf32", b1, "\ntar fp32", a2, "\n    tf32", b2)
    same = (adv0 == adv1).float().mean().item()
    print("identical perturbed elements fp32 vs tf32:", same)
    assert abs(a1["acc"] - b1["acc"]) < 0.005 and abs(a1["miou"] - b1["miou"]) < 0.005
    assert abs(a2["acc"] - b2["acc"]) < 0.005 and abs(a2["miou"] - b2["miou"]) < 0.005
    assert abs((a2["target_acc"] or 0) - (b2["target_acc"] or 0)) < 0.005
    assert a1["acc"] < 0.9                                   # the attack did something
