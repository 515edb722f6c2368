#!/usr/bin/env python
"""A/B of library options at the bench configuration (config[1]: SSG tar-NB, B=16 x 4096, K steps): median attack time
over repeats (CUDA events, L2 flushed) and the per-family times, per option setting.
  python tools/ab_options.py sa_compact=1 sa_compact=0 fps_cluster=0,nn_grid=1"""
import ctypes as C, json, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from pointsecguard_b200 import _lib as L, synthetic as syn, torchattacks
from pointsecguard_b200.engine import MLP_TF32
from pointsecguard_b200.models.pointnet2_sem_seg import get_model

K = int(os.environ.get("AB_STEPS", "50"))
DEFAULTS = {"nn_grid": 0, "fps_cluster": 1, "sa_compact": 1, "x3_fused": 3}
m = get_model(13); m.load_state_dict(syn.make_state_dict("ssg", init="he")); m = m.cuda().eval(); m.set_mlp_mode(int(os.environ.get("AB_MODE", MLP_TF32)))
x, labels, mask = bench.make_inputs(16, 0)
lab = labels.numpy().astype(np.float64)
xd = x.cuda()
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
atk = torchattacks.tar_NB_attack(m, eps=0.5, alpha=0.1, iters=K, target=7, mask=mask)
ref = None
for setting in sys.argv[1:] or ["sa_compact=1", "sa_compact=0"]:
    opts = dict(DEFAULTS)
    opts.update({k: int(v) for k, v in (kv.split("=") for kv in setting.split(","))})
    for k, v in opts.items():
        assert L.psg_set_option(k.encode(), v) == 0, k
    torch.manual_seed(0); out = atk(xd, lab); torch.cuda.synchronize()
    if ref is None:
        ref = out
    same = bool(torch.equal(out, ref))
    ts = []
    for _ in range(7):
        torch.manual_seed(0); flush.fill_(1); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); atk(xd, lab); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    L.psg_prof_enable(1)
    torch.manual_seed(0); atk(xd, lab); torch.cuda.synchronize()
    n = L.psg_prof_ncat(); ms = (C.c_double * n)(); cnt = (C.c_int64 * n)()
    L.psg_prof_collect(ms, cnt); L.psg_prof_enable(0)
    fam = {L.psg_prof_name(i).decode(): round(ms[i] / K, 4) for i in range(n) if cnt[i] and ms[i] / K >= 0.002}
    med = float(np.median(ts))
    print(f"{setting}: {med:.3f} ms per attack ({K * 1e3 / med:.0f} steps/s; min {min(ts):.3f}), identical to first setting: {same}")
    print("   ", json.dumps(fam))
for k, v in DEFAULTS.items():
    L.psg_set_option(k.encode(), v)
