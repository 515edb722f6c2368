"""GPU tests of the API-surface rows that the sem-seg attack path itself never executes (SURVEY.md a6, a11) and of the
1-D-mask batch behaviour of tar_NB_attack."""
import os

import numpy as np
import pytest
import torch

from pointsecguard_b200 import synthetic as syn

pytestmark = pytest.mark.gpu


def _inputs():
    g = torch.Generator("cpu").manual_seed(31)          # oracle/make_golden_misc.py
    xyz = torch.rand(2, 64, 3, generator=g)
    pts = torch.rand(2, 64, 5, generator=g)
    logits = torch.randn(2 * 64, 13, generator=g)
    target = torch.randint(0, 13, (2 * 64,), generator=g)
    weight = torch.rand(13, generator=g) + 0.5
    return xyz, pts, logits, target, weight


def test_sample_and_group_all_vs_reference(golden_dir):
    from pointsecguard_b200.models.pointnet_util import sample_and_group_all
    g = np.load(os.path.join(golden_dir, "api_misc.npz"))
    xyz, pts, *_ = _inputs()
    nx, npts = sample_and_group_all(xyz.cuda(), pts.cuda())
    assert nx.is_cuda and np.array_equal(nx.cpu().numpy(), g["sga_new_xyz"]) and np.array_equal(npts.cpu().numpy(), g["sga_new_points"])
    _, npts2 = sample_and_group_all(xyz.cuda(), None)
    assert np.array_equal(npts2.cpu().numpy(), g["sga_new_points_noattr"])


@pytest.mark.parametrize("arch", ["ssg", "msg"])
def test_get_loss_vs_reference(golden_dir, arch):
    if arch == "ssg":
        from pointsecguard_b200.models.pointnet2_sem_seg import get_loss
    else:
        from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_loss
    g = np.load(os.path.join(golden_dir, "api_misc.npz"))
    _, _, logits, target, weight = _inputs()
    pred = torch.log_softmax(logits, 1).cuda().requires_grad_(True)
    loss = get_loss()(pred, target.cuda(), None, weight.cuda())
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) < 1e-5 * abs(float(g["loss"]))
    np.testing.assert_allclose(pred.grad.cpu().numpy(), g["dpred"], rtol=1e-5, atol=1e-8)


def _ssg():
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    m = get_model(13)
    m.load_state_dict(syn.load_checkpoint("ssg"))
    return m.cuda().eval()


def test_tar_nb_1d_mask_on_a_batch_attacks_block_0_only():
    """target.py:26,36: the reference's cost reads outputs[0], so with a [N] mask and B > 1 only block 0 moves."""
    from pointsecguard_b200 import torchattacks
    m = _ssg()
    x, labels = syn.make_painted_blocks(3, 2048, 2)
    xd = x.cuda()
    mask1 = (labels[0] == 11).numpy()
    lab = labels.numpy().astype(np.float64)
    torch.manual_seed(0)
    adv = torchattacks.tar_NB_attack(m, eps=0.5, alpha=0.1, iters=3, target=7, mask=mask1)(xd, lab)
    assert torch.equal(adv[1:], xd[1:])
    moved = (adv[0, 3:6] != xd[0, 3:6]).any(0).cpu().numpy()
    assert moved[mask1].mean() > 0.9 and not moved[~mask1].any()
    # ... and block 0 moves exactly as it does alone (the draws of a batch of 3 differ from those of a batch of 1, so
    # compare with the same call on a [B,N] mask that is empty for the other blocks)
    mask2 = torch.zeros(3, 2048, dtype=torch.bool)
    mask2[0] = torch.from_numpy(mask1)
    torch.manual_seed(0)
    adv2 = torchattacks.tar_NB_attack(m, eps=0.5, alpha=0.1, iters=3, target=7, mask=mask2)(xd, lab)
    assert torch.equal(adv, adv2)


def test_tar_nb_leaves_unmasked_points_unclamped():
    """target.py:41-43 touches masked points only: colours outside [0,1] elsewhere stay as they are."""
    from pointsecguard_b200 import torchattacks
    m = _ssg()
    x, labels = syn.make_painted_blocks(1, 2048, 5)
    x = x.clone()
    mask = (labels[0] == 11).numpy()
    far = np.where(~mask)[0][:50]
    x[0, 3, far] = 1.7
    x[0, 4, far] = -0.4
    xd = x.cuda()
    torch.manual_seed(0)
    adv = torchattacks.tar_NB_attack(m, eps=0.5, alpha=0.1, iters=3, target=7, mask=mask)(xd, labels.numpy().astype(np.float64))
    assert torch.equal(adv[0, :, far], xd[0, :, far])
    # the model input of the next forward kept them too: a clean forward of adv equals a forward where they were never clamped
    assert float(adv[0, 3, far].max()) == pytest.approx(1.7)

