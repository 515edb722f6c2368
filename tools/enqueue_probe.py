import os, sys, time, torch, numpy as np
sys.path.insert(0, os.getcwd())
from pointsecguard_b200 import synthetic as syn, torchattacks
from pointsecguard_b200.engine import MLP_TF32
from pointsecguard_b200.models.pointnet2_sem_seg import get_model
m = get_model(13); m.load_state_dict(syn.make_state_dict("ssg")); m = m.cuda().eval(); m.set_mlp_mode(MLP_TF32)
x = syn.make_blocks(16, 4096, 0).cuda(); lab = syn.zband_labels(x.cpu()); mask = lab == 11
atk = torchattacks.tar_NB_attack(m, eps=0.5, alpha=0.1, iters=50, target=7, mask=mask)
ln = lab.numpy().astype(np.float64)
for _ in range(2): atk(x, ln)
torch.cuda.synchronize()
from pointsecguard_b200 import _lib as L
l0 = L.psg_launch_count()
t0 = time.perf_counter(); adv = atk(x, ln); t1 = time.perf_counter(); torch.cuda.synchronize(); t2 = time.perf_counter()
print("enqueue ms", (t1 - t0) * 1e3, "total ms", (t2 - t0) * 1e3, "launches", L.psg_launch_count() - l0)
