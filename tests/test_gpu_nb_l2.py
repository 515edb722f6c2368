"""L2-bounded NB / tar-NB on the GPU (``norm="L2"``: csrc/elementwise.cu, pgd_l2_update_kernel; psg_net_pgd_update_l2,
psg_nb_attack_l2).

  * the update kernel alone, in every MLP mode, against the restatement of tests/l2_reference.py (l2_step) built from
    the engine's own read-back gradient: the same fp32 element ops and fp64 norms, so the bits agree;
  * whole attacks against the CPU oracle on the trained checkpoint (per-block relative L2 error of adv - x);
  * the invariants at the bench size (norm bounds, [0, 1], untouched points, run-to-run identity, the target hit-rate);
  * per-block independence from the rest of the batch, sharding, the geometry head start and geometry chunking;
  * the L-inf path is unchanged by the new argument.
"""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import pointnet2_oracle as PO
from pointsecguard_b200 import synthetic as syn

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))      # tests/l2_reference.py
import l2_reference as R  # noqa: E402

pytestmark = pytest.mark.gpu

ORIGIN, TARGET = 11, 7
_MODELS = {}


def _model(arch="ssg", mode="fp32"):
    from pointsecguard_b200.engine import MLP_FP32, MLP_TF32, MLP_TF32X3
    if arch not in _MODELS:
        if arch == "ssg":
            from pointsecguard_b200.models.pointnet2_sem_seg import get_model
        else:
            from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_model
        m = get_model(13)
        m.load_state_dict(syn.load_checkpoint(arch))
        _MODELS[arch] = m.cuda().eval()
    m = _MODELS[arch]
    m.set_mlp_mode({"fp32": MLP_FP32, "tf32": MLP_TF32, "x3": MLP_TF32X3}[mode])
    m.set_shard(None)
    return m


def _ulps(a, b):
    """Distance in units in the last place between two float32 arrays (+0 and -0 coincide)."""
    def key(v):
        i = np.ascontiguousarray(v, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(key(a) - key(b))


def _check_bits(got, want, what):
    d = _ulps(got, want)
    same = float((d == 0).mean()) if d.size else 1.0
    assert same >= 0.9999 and (d.max() if d.size else 0) <= 1, (what, same, d.max())
    return same


# ------------------------------------------------------------------------------------------------------------------
# the update kernel
# ------------------------------------------------------------------------------------------------------------------
SHAPES = [(1, 1100), (5, 1100), (1, 4096), (5, 4096), (1, 16384), (5, 16384), (1, 65536)]


@pytest.mark.parametrize("masked", [False, True], ids=["all", "mask"])
@pytest.mark.parametrize("B, N", SHAPES)
@pytest.mark.parametrize("mode", ["fp32", "x3", "tf32"])
def test_update_kernel_vs_restatement(mode, B, N, masked):
    m = _model("ssg", mode)
    dev = torch.device("cuda")
    x, labels = syn.make_painted_blocks(B, N, 2)
    x = x.contiguous()
    gen = torch.Generator().manual_seed(B * N)
    ori = x[:, 3:6].clone()
    # colours entering the step: a perturbation of the clean ones, so that the projection fires on some blocks only
    cur = torch.clamp(ori + 0.02 * torch.randn(ori.shape, generator=gen), 0, 1)
    xin = x.clone()
    xin[:, 3:6] = cur
    mask = None
    if masked:
        mask = torch.rand(B, N, generator=gen) < 0.3
        if B > 1:
            mask[1] = False                                  # a block with no moving point
    zero_block = 2 if B > 1 else None
    eng = m.engine(dev)
    eng.bind(B, N, 1)
    eng.set_xyz_grad(False)
    eng.set_input(xin.cuda())
    torch.manual_seed(0)
    eng.geometry(eng.draw_starts(1))
    eng.forward(0, True, False)
    dlogp = -torch.nn.functional.one_hot(labels, 13).float() / N          # d(sum CE / N) / d logp
    if zero_block is not None:
        dlogp[zero_block] = 0                                               # a zero-gradient block
    eng.loss_grad_generic(dlogp.cuda())
    g = eng.backward(0, True).cpu()[:, 3:6]
    eps = float(0.02 * np.sqrt(3 * N * (0.3 if masked else 1.0)))         # about the norm of the perturbation of cur
    alpha = 0.5 * eps
    msk = mask.to(torch.uint8).cuda() if mask is not None else None
    adv = xin.clone().cuda()
    eng.pgd_update_l2(adv, ori.cuda(), msk, 3, 3, alpha, eps)
    # the projected colours the update left in the model input: a second update at alpha = 0 writes adv = cur
    col = xin.clone().cuda()
    eng.pgd_update_l2(col, ori.cuda(), msk, 3, 3, 0.0, eps)
    torch.cuda.synchronize()
    adv, col = adv.cpu(), col.cpu()

    moving = torch.ones(B, 1, N, dtype=torch.bool) if mask is None else mask.view(B, 1, N)
    a_ref, col_ref = R.l2_step(cur, ori, g * moving, alpha, eps, moving)
    mv3 = moving.expand(B, 3, N)
    s_adv = _check_bits(adv[:, 3:6][mv3].numpy(), a_ref[mv3].numpy(), "adv")
    s_col = _check_bits(col[:, 3:6][mv3].numpy(), col_ref[mv3].numpy(), "projected colours")
    # nothing else is read or written
    assert torch.equal(adv[:, :3], xin[:, :3]) and torch.equal(adv[:, 6:], xin[:, 6:])
    assert torch.equal(adv[:, 3:6][~mv3], xin[:, 3:6][~mv3]) and torch.equal(col[:, 3:6][~mv3], xin[:, 3:6][~mv3])
    assert not torch.isnan(adv).any() and not torch.isnan(col).any()
    if zero_block is not None:
        assert torch.equal(g[zero_block], torch.zeros_like(g[zero_block]))
        assert torch.equal(adv[zero_block], xin[zero_block])
    dn = ((col[:, 3:6] - ori) * mv3).double().pow(2).flatten(1).sum(1).sqrt()
    assert (dn <= eps * (1 + 1e-6)).all() and (col[:, 3:6] >= 0).all() and (col[:, 3:6] <= 1).all()
    fired = int(((a_ref - ori) * mv3).double().pow(2).flatten(1).sum(1).sqrt().gt(eps).sum())
    print(f"L2 update {mode} B={B} N={N} mask={masked}: adv identical {s_adv:.6f}, projected colours identical {s_col:.6f}, "
          f"projection fired on {fired} of {B} blocks")


def test_update_rejects_bad_arguments():
    from pointsecguard_b200 import _lib as L
    m = _model("ssg", "fp32")
    eng = m.engine(torch.device("cuda"))
    eng.bind(1, 1024, 1)
    adv = torch.zeros(1, 9, 1024, device="cuda")
    ori = torch.zeros(1, 3, 1024, device="cuda")
    for c0, nc, alpha, eps in ((3, 3, 0.1, -1.0), (3, 3, float("nan"), 1.0), (3, 3, 0.1, float("inf")), (7, 3, 0.1, 1.0),
                               (3, 0, 0.1, 1.0)):
        with pytest.raises(L.PsgError):
            eng.pgd_update_l2(adv, ori, None, c0, nc, alpha, eps)
    with pytest.raises(ValueError):
        eng.nb_attack(adv, ori, None, None, 7, 1, 0, 0.1, 1.0, 1.0, norm="L1")


# ------------------------------------------------------------------------------------------------------------------
# whole attacks against the CPU oracle
# ------------------------------------------------------------------------------------------------------------------
_ORACLE = {}
EPS, ALPHA = 1.0, 0.5          # |adv - x| reaches 1.35-1.8 in five steps (oracle): the projection fires in the 5-step runs


def _cases():
    x2, l2 = syn.make_painted_blocks(2, 2048, 0)
    x1, l1 = syn.make_painted_blocks(1, 2048, 1)
    return {"nb": (x2, l2, None), "tar_mask1d": (x1, l1, (l1[0] == ORIGIN).numpy()), "tar_maskBN": (x2, l2, l2 == ORIGIN)}


def _oracle(arch, case, iters):
    """The oracle's adv after ``iters`` iterations and the projected colours entering each of them."""
    key = (arch, case, iters)
    if key not in _ORACLE:
        x, labels, mask = _cases()[case]
        om = PO.OracleModel(syn.load_checkpoint(arch), arch)
        snaps = []
        torch.manual_seed(0)
        if mask is None:
            adv = R.nb_attack_l2(om, x, labels.numpy().astype(np.float64), eps=EPS, alpha=ALPHA, iters=iters,
                                 snapshots=snaps)
        else:
            adv = R.tar_nb_attack_l2(om, x, eps=EPS, alpha=ALPHA, iters=iters, target=TARGET, mask=mask,
                                     snapshots=snaps)
        _ORACLE[key] = (adv, snaps)
    return _ORACLE[key]


def _gpu(m, case, iters, x=None, skip=0):
    """The package's attack; ``x`` replaces the case's input and ``skip`` forwards' FPS draws are consumed first."""
    from pointsecguard_b200 import distributed as D, torchattacks
    x0, labels, mask = _cases()[case]
    x = x0 if x is None else x
    B, _, N = x.shape
    torch.manual_seed(0)
    if skip:
        D.draw_starts([N, 1024, 256, 64], skip, D.Shard(B, 0, B))
    if mask is None:
        atk = torchattacks.NB_attack(m, eps=EPS, alpha=ALPHA, iters=iters, norm="L2")
    else:
        atk = torchattacks.tar_NB_attack(m, eps=EPS, alpha=ALPHA, iters=iters, target=TARGET, mask=mask, norm="L2")
    return atk(x.cuda(), labels.numpy().astype(np.float64)).cpu()


def _rel(adv, ref, x):
    d, r = (adv - x)[:, 3:6].double(), (ref - x)[:, 3:6].double()
    return ((d - r).flatten(1).norm(dim=1) / r.flatten(1).norm(dim=1)).numpy(), (d - r).pow(2).sum(1), r


def _fmt(rel):
    return "[" + " ".join(f"{v:.2e}" for v in rel) + "]"


def _flip_only(err2, r, b, gate):
    """A block that misses the gate because of a discrete flip (max-pool arg-max / ReLU near a tie) carries its error on a
    few points: without its 1 % worst points the block is within the gate."""
    k = max(1, err2.shape[1] // 100)
    keep = torch.ones(err2.shape[1], dtype=torch.bool)
    keep[err2[b].topk(k).indices] = False
    rest = float(err2[b][keep].sum().sqrt() / r[b].flatten().norm())
    share = float(err2[b][~keep].sum() / err2[b].sum())
    print(f"    block {b}: {share:.3f} of the squared error on its {k} worst points; the rest {rest:.2e}")
    return rest <= gate


@pytest.mark.parametrize("case", ["nb", "tar_mask1d", "tar_maskBN"])
@pytest.mark.parametrize("arch", ["ssg", "msg"])
@pytest.mark.parametrize("mode", ["fp32", "x3", "tf32"])
def test_attack_vs_oracle(mode, arch, case):
    """Per-block relative L2 error of adv - x against the oracle.  After 5 iterations a block that misses the gate is
    replayed from the oracle's colours entering its last iteration, with that forward's FPS draws (the last-step replay of
    test_gpu_configs.py): one step from the same state must meet the gate.  A block whose error sits on a flip (its 1 %
    worst points) is shown as such and must meet the gate on its other points.
    Measured on a B200 (fp32 / 3xTF32): most blocks agree to 1e-6 after one step, single blocks reach 3e-4 (fp32) and
    9e-4 (3xTF32), and a 3xTF32 block with 98 % of its error on 20 points (a flip) 4.5e-3, 5.9e-4 without them.  Replayed
    fifth steps: up to 4.5e-4 in one run; 3.4e-3, and 2e-2 with 6.9e-3 off the flip, in a run on another machine (the
    CPU oracle's sums follow the host's thread count, so its trajectory differs near a tie).  The gates are therefore
    1e-3 (one step) and 1e-2 (replayed fifth step) outside flips."""
    m = _model(arch, mode)
    x = _cases()[case][0]
    gates = {1: 1e-3, 5: 1e-2} if mode != "tf32" else {1: 0.25}
    for iters, gate in gates.items():
        adv = _gpu(m, case, iters)
        ref, snaps = _oracle(arch, case, iters)
        rel, err2, r = _rel(adv, ref, x)
        print(f"L2 attack {mode} {arch} {case} {iters} it: per-block relative error of adv - x {_fmt(rel)}")
        assert torch.equal(adv[:, :3], x[:, :3]) and torch.equal(adv[:, 6:], x[:, 6:])
        miss = [b for b in range(len(rel)) if not rel[b] <= gate]
        if miss and iters > 1:
            mask = _cases()[case][2]
            B, _, N = x.shape
            mv = torch.ones(B, 1, N, dtype=torch.bool) if mask is None else \
                torch.as_tensor(np.asarray(mask)).view(-1, 1, N).expand(B, 1, N)
            x2 = x.clone()
            x2[:, 3:6] = torch.where(mv, snaps[-1], x[:, 3:6])
            rel, err2, r = _rel(_gpu(m, case, 1, x2, skip=iters - 1), ref, x2)
            print(f"    last-step replay: per-block relative error of the step {_fmt(rel)}")
            miss = [b for b in range(len(rel)) if not rel[b] <= gate]
        for b in miss:
            assert _flip_only(err2, r, b, gate), (iters, b, rel, gate)


# ------------------------------------------------------------------------------------------------------------------
# invariants at the bench size: B = 16 blocks of 4096 points, 50 iterations
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_invariants_at_bench_size(mode):
    from pointsecguard_b200 import metrics as MT, torchattacks
    m = _model("ssg", mode)
    x, labels = syn.make_painted_blocks(16, 4096, 0)
    mask = labels == ORIGIN
    xd = x.cuda()
    eps, alpha = 2.0, 0.25
    runs = []
    for head in (None, None, 0):
        if head is not None:
            m.geometry_head = head          # the last run's final update is on the primary engine: read its colours back
        torch.manual_seed(0)
        atk = torchattacks.tar_NB_attack(m, eps=eps, alpha=alpha, iters=50, target=TARGET, mask=mask.numpy(), norm="L2")
        runs.append(atk(xd, labels.numpy().astype(np.float64)))
    del m.geometry_head
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2])
    # the colours the last update projected (the model input it left behind), read back by an update at alpha = 0
    eng = m.engine(xd.device)
    buf = xd.clone().contiguous()
    eng.pgd_update_l2(buf, xd[:, 3:6].contiguous(), mask.to(torch.uint8).cuda(), 3, 3, 0.0, eps)
    col = buf.cpu()[:, 3:6]
    adv = runs[0].cpu()
    mv = mask.view(16, 1, 4096)
    mv3 = mv.expand(16, 3, 4096)
    assert torch.equal(adv[:, :3], x[:, :3]) and torch.equal(adv[:, 6:], x[:, 6:])
    assert torch.equal(adv[:, 3:6][~mv3], x[:, 3:6][~mv3])
    dn = ((adv[:, 3:6] - x[:, 3:6]).double() * mv).flatten(1).norm(dim=1)
    cn = ((col - x[:, 3:6]).double() * mv).flatten(1).norm(dim=1)
    assert (dn <= (eps + alpha) * (1 + 1e-6)).all()
    assert (cn <= eps * (1 + 1e-6)).all() and (col >= 0).all() and (col <= 1).all()

    def hit_rate(inp):
        torch.manual_seed(1)
        with torch.no_grad():
            logp, _ = m(inp)
        return MT.summarize(MT.attack_counters(logp, labels.cuda(), mask.cuda(), TARGET).cpu(), 13)["target_acc"]

    clean, attacked = hit_rate(xd), hit_rate(runs[0])            # the scripts evaluate the returned (un-projected) tensor
    print(f"L2 tar-NB {mode} B=16 N=4096 50 it eps={eps} alpha={alpha}: target hit-rate clean {clean:.4f} -> attacked "
          f"{attacked:.4f}; |adv - x| per block max {dn.max().item():.4f}, |col - x| max {cn.max().item():.4f}")
    assert attacked > clean


# ------------------------------------------------------------------------------------------------------------------
# independence from the rest of the batch, sharding, the head start and chunking
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("targeted", [False, True], ids=["nb", "tar_nb"])
def test_shard_matches_the_blocks_of_the_whole_batch(targeted):
    from pointsecguard_b200 import torchattacks
    from pointsecguard_b200.distributed import Shard
    m = _model("ssg", "fp32")
    x, labels = syn.make_painted_blocks(4, 2048, 3)
    mask = labels == ORIGIN

    def run(sl):
        torch.manual_seed(0)
        if targeted:
            atk = torchattacks.tar_NB_attack(m, eps=EPS, alpha=ALPHA, iters=10, target=TARGET, mask=mask[sl], norm="L2")
        else:
            atk = torchattacks.NB_attack(m, eps=EPS, alpha=ALPHA, iters=10, norm="L2")
        return atk(x[sl].cuda(), labels[sl].numpy().astype(np.float64)).cpu()

    whole = run(slice(0, 4))
    m.set_shard(Shard(4, 2, 2))
    try:
        part = run(slice(2, 4))
    finally:
        m.set_shard(None)
    assert not torch.equal(whole[2:], x[2:])
    assert torch.equal(whole[2:], part)


def test_head_start_and_chunking_do_not_change_the_result(monkeypatch):
    from pointsecguard_b200 import torchattacks
    from pointsecguard_b200.torchattacks.attacks import nontarget
    m = _model("ssg", "fp32")
    x, labels = syn.make_painted_blocks(8, 2048, 4)
    lab = labels.numpy().astype(np.float64)
    xd = x.cuda()

    def run(iters):
        torch.manual_seed(0)
        return torchattacks.NB_attack(m, eps=EPS, alpha=0.1, iters=iters, norm="L2")(xd, lab)

    head = run(20)                          # geometry head start on (the default of 4 forwards)
    m.geometry_head = 0
    try:
        plain = run(20)
    finally:
        del m.geometry_head
    assert torch.equal(head, plain)

    two_chunks = run(130)                   # 1024 // 8 = 128 forwards of geometry per chunk: two chunks
    monkeypatch.setattr(nontarget, "_MAX_PROBLEMS", 8 * 130)
    one_chunk = run(130)
    assert torch.equal(two_chunks, one_chunk)


@pytest.mark.parametrize("targeted", [False, True], ids=["nb", "tar_nb"])
def test_linf_argument_is_the_default(targeted):
    from pointsecguard_b200 import torchattacks
    m = _model("ssg", "fp32")
    x, labels = syn.make_painted_blocks(2, 2048, 5)
    kw = dict(target=TARGET, mask=(labels == ORIGIN).numpy()) if targeted else {}
    cls = torchattacks.tar_NB_attack if targeted else torchattacks.NB_attack
    out = []
    for extra in ({}, {"norm": "Linf"}):
        torch.manual_seed(0)
        out.append(cls(m, eps=0.1, alpha=0.05, iters=5, **kw, **extra)(x.cuda(), labels.numpy().astype(np.float64)))
    assert torch.equal(out[0], out[1])
