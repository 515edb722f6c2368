#!/usr/bin/env python
"""A/B of library options on BASELINE config 3 (MSG NB, B = 64 x 4096, 10 iterations): time per attack per option setting.
  python tools/ab_msg.py sa_compact=1 sa_compact=0"""
import ctypes as C, json, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointsecguard_b200 import _lib as L, synthetic as syn, torchattacks
from pointsecguard_b200.engine import MLP_TF32
from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_model

for kv in filter(None, os.environ.get("AB_PRE", "").split(",")):        # options that must be set before the engine is bound
    k, v = kv.split("="); assert L.psg_set_option(k.encode(), int(v)) == 0, k
m = get_model(13); m.load_state_dict(syn.make_state_dict("msg", init="he")); m = m.cuda().eval(); m.set_mlp_mode(int(os.environ.get("AB_MODE", MLP_TF32)))
B = int(os.environ.get("AB_BLOCKS", "64"))
x = syn.make_blocks(B, 4096, 0).cuda(); torch.manual_seed(5); lab = m(x)[0].argmax(2).cpu().numpy().astype(np.float64)
atk = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=10)
ref = None
for setting in sys.argv[1:] or ["sa_compact=1", "sa_compact=0"]:
    for kv in setting.split(","):
        k, v = kv.split("="); assert L.psg_set_option(k.encode(), int(v)) == 0, k
    torch.manual_seed(0); out = atk(x, lab); torch.cuda.synchronize()
    ref = out if ref is None else ref
    ts = []
    for _ in range(5):
        torch.manual_seed(0); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); atk(x, lab); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    L.psg_prof_enable(1); torch.manual_seed(0); atk(x, lab); torch.cuda.synchronize()
    n = L.psg_prof_ncat(); ms = (C.c_double * n)(); cnt = (C.c_int64 * n)(); L.psg_prof_collect(ms, cnt); L.psg_prof_enable(0)
    fam = {L.psg_prof_name(i).decode(): round(ms[i] / 10, 4) for i in range(n) if cnt[i] and ms[i] / 10 >= 0.01}
    print(f"{setting}: {np.median(ts):.3f} ms per attack ({10e3 / np.median(ts):.1f} steps/s), identical to first: {bool(torch.equal(out, ref))}")
    print("   ", json.dumps(fam))
