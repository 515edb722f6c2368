"""GPU parity of the whole network (forward log-probabilities, l4 features, input gradient) and of
the NB / tar-NB attack loops against the golden vectors of the executed reference and the CPU
oracle.  Tolerances (stated, fp32 MLP mode): log-probabilities rtol 1e-3 / atol 1e-4; colour
gradient relative Frobenius error < 1e-2 with sign agreement > 99.9 % (the oracle's own fp32 vs
fp64 gradient differs by 5.9e-3, SURVEY.md App. B); perturbed colours identical on > 99.5 % of the
elements (a flipped sign is a 2*alpha jump)."""
import os

import numpy as np
import pytest
import torch

from pointsecguard_b200 import synthetic as syn

pytestmark = pytest.mark.gpu


def _model(arch, mode=0):
    if arch == "ssg":
        from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    else:
        from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_model
    m = get_model(13)
    m.load_state_dict(syn.make_state_dict(arch))
    m = m.cuda().eval()
    m.set_mlp_mode(mode)          # 0: fp32 CUDA cores; 2: error-compensated 3xTF32 on tcgen05 -- both held to the fp32 gates
    return m


def _grad_report(mine, ref):
    rel = np.linalg.norm(mine - ref) / np.linalg.norm(ref)
    nz = ref != 0
    sign = (np.sign(mine[nz]) == np.sign(ref[nz])).mean()
    close = (np.abs(mine - ref) <= 1e-3 * np.abs(ref) + 1e-12).mean()
    return rel, sign, close


@pytest.mark.parametrize("mode", [0, 2], ids=["fp32", "x3"])
@pytest.mark.parametrize("arch", ["ssg", "msg"])
def test_forward_and_input_gradient_vs_reference_golden(golden_dir, arch, mode):
    g = dict(np.load(os.path.join(golden_dir, f"model_{arch}.npz")))
    m = _model(arch, mode)
    x = syn.make_blocks(2, 2048, 0, "uniform").cuda().requires_grad_(True)
    torch.manual_seed(0)
    logp, l4 = m(x)
    assert logp.shape == (2, 2048, 13) and l4.shape == g["l4"].shape
    np.testing.assert_allclose(logp.detach().cpu().numpy(), g["logp"], rtol=1e-3, atol=1e-4)
    np.testing.assert_allclose(l4.cpu().numpy(), g["l4"], rtol=1e-3, atol=1e-4)
    assert (logp.detach().cpu().numpy().argmax(2) == g["logp"].argmax(2)).mean() > 0.999
    y = torch.from_numpy(g["y"]).long().cuda()
    cost = torch.nn.functional.cross_entropy(logp.reshape(-1, 13), y.view(-1), reduction="sum") / logp.size(1)
    cost.backward()
    mine = x.grad.cpu().numpy()
    # colour (3:6) and normalised-xyz (6:9) channels reach the loss through features only
    rel, sign, close = _grad_report(mine[:, 3:], g["grad"][:, 3:])
    print(f"{arch}: grad rel={rel:.2e} sign={sign:.5f} within-rtol-1e-3={close:.4f}")
    # SURVEY section 7, hard part 2: >= 99.9 % of the elements within rtol 1e-3, sign agreement >= 99.99 %.  Measured: fp32
    # rel 3.4e-6 / 1.8e-6, within rtol 0.9998 / 1.0000; 3xTF32 rel 4.5e-6 / 1.8e-5, within rtol 0.9998 / 0.9997 (8e-4 / 1.2e-3
    # and 0.9988 / 0.9973 before the accumulator-truncation bias was folded into its weights); sign 1.00000 everywhere
    assert rel < 1e-4 and sign >= 0.9999
    assert close >= 0.999


def test_engine_indices_match_reference_trace(golden_dir):
    """The FPS / ball-query indices the engine computes inside a forward are the reference's."""
    from pointsecguard_b200.models import pointnet_util as PU
    g = dict(np.load(os.path.join(golden_dir, "model_ssg.npz")))
    ref = [g[k] for k in sorted(k for k in g if k.startswith("idx"))]   # fps, ball per level
    x = syn.make_blocks(2, 2048, 0, "uniform").cuda()
    xyz = x[:, :3].permute(0, 2, 1).contiguous()
    torch.manual_seed(0)
    cfg = [(1024, 0.1, 32), (256, 0.2, 32), (64, 0.4, 32), (16, 0.8, 32)]
    k = 0
    for S, r, K in cfg:
        fps = PU.farthest_point_sample(xyz, S)
        assert np.array_equal(fps.cpu().numpy(), ref[k]); k += 1
        new_xyz = PU.index_points(xyz, fps)
        idx = PU.query_ball_point(r, K, xyz, new_xyz)
        assert np.array_equal(idx.cpu().numpy(), ref[k]); k += 1
        xyz = new_xyz


def test_backward_needs_latest_forward():
    m = _model("ssg")
    x = syn.make_blocks(1, 1024, 0).cuda().requires_grad_(True)
    logp, _ = m(x)
    m(x.detach())
    with pytest.raises(RuntimeError):
        logp.sum().backward()


def test_cpu_tensors_are_refused_in_both_modes():
    m = _model("ssg")
    with pytest.raises(RuntimeError):
        m.train()(syn.make_blocks(1, 1024, 0))
    with pytest.raises(RuntimeError):
        m.eval()(syn.make_blocks(1, 1024, 0))


@pytest.mark.parametrize("mode", [0, 2], ids=["fp32", "x3"])
def test_nb_attack_vs_reference_golden(golden_dir, mode):
    from pointsecguard_b200 import torchattacks
    g = dict(np.load(os.path.join(golden_dir, "attack.npz")))
    m = _model("ssg", mode)
    x = syn.make_blocks(2, 4096, 0, "uniform").cuda()
    torch.manual_seed(0)
    adv = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=3)(x, g["nb_labels"].astype(np.float64))
    assert adv.shape == x.shape
    assert torch.equal(adv[:, :3], x[:, :3]) and torch.equal(adv[:, 6:], x[:, 6:])
    same = (adv[:, 3:6].cpu().numpy() == g["nb_adv"]).mean()
    print("NB identical fraction", same)
    assert same > 0.995
    dev = (adv[:, 3:6] - x[:, 3:6]).abs().max().item()
    assert 0.1 < dev <= 0.15 + 1e-6                 # Q1: un-projected last step is returned


def test_tar_nb_attack_vs_reference_golden(golden_dir):
    from pointsecguard_b200 import torchattacks
    g = dict(np.load(os.path.join(golden_dir, "attack.npz")))
    m = _model("ssg")
    x1 = syn.make_blocks(1, 4096, 1, "uniform").cuda()
    zl = syn.zband_labels(x1.cpu())
    mask = (zl[0] == 11).numpy()
    torch.manual_seed(0)
    adv = torchattacks.tar_NB_attack(m, eps=0.5, alpha=0.1, iters=3, target=7, mask=mask)(x1, zl.numpy().astype(np.float64))
    same = (adv[:, 3:6].cpu().numpy() == g["tnb_adv"]).mean()
    print("tar-NB identical fraction", same)
    assert same > 0.995
    unmasked = ~torch.from_numpy(mask)
    assert torch.equal(adv[0, 3:6][:, unmasked].cpu(), x1[0, 3:6][:, unmasked].cpu())


def test_msg_nb_attack_vs_reference_golden(golden_dir):
    from pointsecguard_b200 import torchattacks
    g = dict(np.load(os.path.join(golden_dir, "attack.npz")))
    m = _model("msg")
    x1 = syn.make_blocks(1, 4096, 1, "uniform").cuda()
    torch.manual_seed(0)
    adv = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=2)(x1, g["msg_nb_labels"].astype(np.float64))
    same = (adv[:, 3:6].cpu().numpy() == g["msg_nb_adv"]).mean()
    print("MSG NB identical fraction", same)
    assert same > 0.995


def test_attack_is_deterministic():
    from pointsecguard_b200 import torchattacks
    m = _model("ssg")
    x = syn.make_blocks(2, 4096, 2).cuda()
    lab = syn.zband_labels(x.cpu()).numpy().astype(np.float64)
    outs = []
    for _ in range(2):
        torch.manual_seed(7)
        outs.append(torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=3)(x, lab))
    assert torch.equal(outs[0], outs[1])            # no float atomics anywhere on the path


def test_tf32_attack_is_run_to_run_deterministic_at_bench_size():
    """The fused tcgen05 path at the bench configuration (16 x 4096, 50 steps), eight runs: bit-identical.  A race
    between the warps of one tile (the pooled scratch of a slow warp overwritten by a fast warp's next gather) used to
    flip a few hundred values in about one run out of three; differences grow over the steps, so the long attack is
    the sensitive probe."""
    from pointsecguard_b200 import torchattacks
    from pointsecguard_b200.engine import MLP_FP32, MLP_TF32
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    m = get_model(13)
    m.load_state_dict(syn.make_state_dict("ssg", init="he"))
    m = m.cuda().eval()
    m.set_mlp_mode(MLP_TF32)
    x = syn.make_blocks(16, 4096, 0)
    labels = syn.zband_labels(x)
    mask = labels == 11
    lab = labels.numpy().astype(np.float64)
    xd = x.cuda()
    first = None
    for _ in range(8):
        torch.manual_seed(0)
        adv = torchattacks.tar_NB_attack(m, eps=0.5, alpha=0.1, iters=50, target=7, mask=mask)(xd, lab)
        if first is None:
            first = adv.clone()
        else:
            assert int((adv != first).sum()) == 0
    m.set_mlp_mode(MLP_FP32)


def test_tf32_msg_attack_is_run_to_run_deterministic():
    """Same probe for the multi-radius network (K = 16 and K = 32 branches of the fused kernels, wide tile programs)."""
    from pointsecguard_b200 import torchattacks
    from pointsecguard_b200.engine import MLP_FP32, MLP_TF32
    from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_model
    m = get_model(13)
    m.load_state_dict(syn.make_state_dict("msg", init="he"))
    m = m.cuda().eval()
    m.set_mlp_mode(MLP_TF32)
    x = syn.make_blocks(8, 4096, 5)
    lab = syn.zband_labels(x).numpy().astype(np.float64)
    xd = x.cuda()
    first = None
    for _ in range(5):
        torch.manual_seed(0)
        adv = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=12)(xd, lab)
        if first is None:
            first = adv.clone()
        else:
            assert int((adv != first).sum()) == 0
    m.set_mlp_mode(MLP_FP32)


def test_sharded_attack_equals_full_batch_attack():
    """Two 'ranks' (run one after the other on this GPU) that each attack their shard of a global batch
    -- FPS starts drawn for the GLOBAL batch and sliced (distributed.py) -- reproduce the full-batch
    attack block for block, bit for bit, and their summed counters equal the full-batch counters."""
    from pointsecguard_b200 import distributed as D, metrics as MT, torchattacks
    m = _model("ssg")
    G = 4
    x = syn.make_blocks(G, 2048, 5).cuda()
    lab_t = syn.zband_labels(x.cpu())
    lab = lab_t.numpy().astype(np.float64)
    torch.manual_seed(3)
    full = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=3)(x, lab)
    torch.manual_seed(4)
    c_full = MT.attack_counters(m(full)[0], lab_t.cuda())
    parts, counters = [], torch.zeros_like(c_full)
    for r in range(2):
        sh = D.shard_for(G, r, 2)
        m.set_shard(sh)
        torch.manual_seed(3)
        adv = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=3)(sh.slice(x), sh.slice(lab))
        torch.manual_seed(4)
        counters += MT.attack_counters(m(adv)[0], sh.slice(lab_t).cuda())
        parts.append(adv)
    m.set_shard(None)
    assert torch.equal(torch.cat(parts), full)
    assert torch.equal(counters, c_full)


@pytest.mark.parametrize("arch", ["ssg", "msg"])
def test_coordinate_gradient_vs_reference_golden(golden_dir, arch):
    """With model.xyz_grad the autograd of forward() is complete on all nine channels: channels 0:3 get
    the gradient through the features AND through the geometry (centred neighbour coordinates of every
    SA level, inverse-distance weights of every FP level), as the reference's autograd computes it."""
    g = dict(np.load(os.path.join(golden_dir, f"model_{arch}.npz")))
    m = _model(arch)
    m.xyz_grad = True
    x = syn.make_blocks(2, 2048, 0, "uniform").cuda().requires_grad_(True)
    torch.manual_seed(0)
    logp, _ = m(x)
    y = torch.from_numpy(g["y"]).long().cuda()
    cost = torch.nn.functional.cross_entropy(logp.reshape(-1, 13), y.view(-1), reduction="sum") / logp.size(1)
    cost.backward()
    mine = x.grad.cpu().numpy()
    rel, sign, close = _grad_report(mine[:, :3], g["grad"][:, :3])
    print(f"{arch}: xyz grad rel={rel:.2e} sign={sign:.5f} within-rtol-1e-3={close:.4f}")
    assert rel < 2e-2 and sign > 0.995
    rel_all, sign_all, _ = _grad_report(mine, g["grad"])
    assert rel_all < 2e-2 and sign_all > 0.998


def test_coordinate_gradient_with_repeated_fps_indices_vs_oracle():
    """A cloud with fewer distinct points than SA1 samples: FPS runs out of distinct points and selects one index many
    times, so xyz_l = xyz_{l-1}[fps_idx] scatters many gradient rows into ONE source point -- the ordered multi-add
    path of fps_xyz_back_kernel -- checked against the CPU autograd of the oracle model."""
    from oracle import pointnet2_oracle as PO
    sd = syn.make_state_dict("ssg")
    m = _model("ssg")
    m.xyz_grad = True
    gen = torch.Generator().manual_seed(3)
    base = syn.make_blocks(1, 1024, 4, "uniform")                       # [1,9,1024]
    pick = torch.randint(0, 600, (1, 1024), generator=gen)              # 1024 points, at most 600 distinct
    x0 = torch.gather(base, 2, pick.unsqueeze(1).expand(1, 9, 1024)).contiguous()
    y = syn.zband_labels(x0).long()
    xo = x0.clone().requires_grad_(True)
    torch.manual_seed(0)
    lo, _ = PO.OracleModel(sd, "ssg")(xo)
    (torch.nn.functional.cross_entropy(lo.reshape(-1, 13), y.view(-1), reduction="sum") / lo.size(1)).backward()
    xg = x0.clone().cuda().requires_grad_(True)
    torch.manual_seed(0)
    lg, _ = m(xg)
    (torch.nn.functional.cross_entropy(lg.reshape(-1, 13), y.view(-1).cuda(), reduction="sum") / lg.size(1)).backward()
    # the engine really saw repeated indices at SA1 (1024 samples out of <= 600 distinct points)
    rel, sign, close = _grad_report(xg.grad.cpu().numpy()[:, :3], xo.grad.numpy()[:, :3])
    print(f"repeated fps indices: xyz grad rel={rel:.2e} sign={sign:.5f} within-rtol-1e-3={close:.4f}")
    # coincident points make many coordinate gradients cancel to ~0 (random sign there), so the gate is the relative error
    assert rel < 1e-3 and sign > 0.95
    rel_all, sign_all, _ = _grad_report(xg.grad.cpu().numpy(), xo.grad.numpy())
    assert rel_all < 1e-3 and sign_all > 0.95


def test_attack_metrics_vs_oracle_within_half_a_point():
    """north_star gate: accuracy and mIoU after N attack iterations agree with the CPU oracle within
    +-0.5 pt.  Uses the input-sensitive synthetic checkpoint (init="he"), on which the attack really
    flips predictions (the default-scale checkpoint predicts one class everywhere)."""
    from oracle import attacks_oracle as AO
    from oracle import pointnet2_oracle as PO
    from pointsecguard_b200 import metrics as MT, torchattacks
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    sd = syn.make_state_dict("ssg", init="he")
    m = get_model(13)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    om = PO.OracleModel(sd, "ssg")
    x = syn.make_blocks(2, 2048, 3)
    torch.manual_seed(5)
    lab = om(x)[0].argmax(2)
    torch.manual_seed(0)
    ref = AO.nb_attack(om, x, lab.numpy().astype(np.float64), eps=0.1, alpha=0.05, iters=5)
    torch.manual_seed(1)
    ref_pred = om(ref)[0].argmax(2)
    ref_m = AO.block_metrics(ref_pred.numpy(), lab.numpy().astype(np.float64))
    torch.manual_seed(0)
    adv = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=5)(x.cuda(), lab.numpy().astype(np.float64))
    torch.manual_seed(1)
    mine = MT.summarize(MT.attack_counters(m(adv)[0], lab.cuda()))
    same = (adv[:, 3:6].cpu() == ref[:, 3:6]).float().mean().item()
    print(f"oracle acc {ref_m['acc']:.4f} miou {ref_m['miou']:.4f} | gpu acc {mine['acc']:.4f} miou {mine['miou']:.4f} | identical {same:.4f}")
    assert ref_m["acc"] < 0.95                                # the attack moved the predictions
    assert abs(mine["acc"] - ref_m["acc"]) < 0.005 and abs(mine["miou"] - ref_m["miou"]) < 0.005
    assert same > 0.99


def test_whole_scene_voting_vs_oracle():
    """SURVEY.md 8f rank 1: add_vote + scene IoU on the GPU against the restated script arithmetic,
    including the scripts' all-zero weight quirk (nothing is voted, scene prediction = class 0)."""
    from oracle import attacks_oracle as AO
    from pointsecguard_b200 import metrics as MT
    rng = np.random.default_rng(0)
    P, B, N = 5000, 4, 1024
    logp = torch.randn(B, N, 13, generator=torch.Generator().manual_seed(0))
    pidx = torch.from_numpy(rng.integers(0, P, (B, N)))
    weight = torch.from_numpy((rng.random((B, N)) < 0.8).astype(np.float32))
    scene_lab = torch.from_numpy(rng.integers(0, 13, P))
    pool_ref = AO.add_vote(np.zeros((P, 13)), pidx.numpy(), logp.argmax(2).numpy(), weight.numpy())
    vp = MT.VotePool(P, 13).add(logp.cuda(), pidx, weight).add(logp.cuda(), pidx, weight)      # two votes
    assert np.array_equal(vp.pool.cpu().numpy(), 2 * pool_ref)
    ref = AO.scene_metrics(pool_ref, scene_lab.numpy())
    got = MT.scene_iou(vp.counters(scene_lab.cuda()))
    assert abs(got["miou_seen"] - ref["miou"]) < 1e-9 and abs(got["acc"] - ref["acc"]) < 1e-6
    # the scripts' own weights are all zero: empty pool, every scene point predicted as class 0
    empty = MT.VotePool(P, 13).add(logp.cuda(), pidx, torch.zeros(B, N))
    assert float(empty.pool.sum()) == 0.0
    c = empty.counters(scene_lab.cuda()).cpu().numpy()[:169].reshape(13, 13)
    assert c[:, 0].sum() == P and c[:, 1:].sum() == 0
