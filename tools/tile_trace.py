#!/usr/bin/env python
"""Phase trace of the tile programs (csrc/chain_fused.cu): clock64 stamps of CTA 0 for every tile-program
launch of ONE attack step at the bench configuration.  Prints, per launch, the time each op spends in
refill (E0), waiting for the accumulator (E1 - E0) and in the epilogue (E2 - E1), plus the MMA issuer's view.

    python tools/tile_trace.py [--blocks 16] > gpurun_out/tile_trace.txt
"""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=16)
    ap.add_argument("--launches", type=int, default=12)
    ap.add_argument("--raw", action="store_true", help="print the raw stamp deltas of every launch (fused SA kernels included)")
    args = ap.parse_args()
    from pointsecguard_b200 import _lib as L
    from pointsecguard_b200 import synthetic as syn, torchattacks
    from pointsecguard_b200.engine import MLP_TF32
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    dev = torch.device("cuda", 0)
    model = get_model(13)
    model.load_state_dict(syn.make_state_dict("ssg", init="he"))
    model = model.to(dev).eval()
    model.set_mlp_mode(MLP_TF32)
    x, labels, mask = bench.make_inputs(args.blocks, 0)
    lab = labels.numpy().astype(np.float64)
    mk = lambda it: torchattacks.tar_NB_attack(model, eps=bench.EPS, alpha=bench.ALPHA, iters=it, target=bench.TARGET, mask=mask)
    xd = x.to(dev)
    mk(5)(xd, lab)
    torch.cuda.synchronize()
    buf = torch.zeros(args.launches, 4, 512, dtype=torch.int64, device=dev)
    L.psg_debug_trace(buf.data_ptr(), args.launches)
    mk(1)(xd, lab)
    torch.cuda.synchronize()
    L.psg_debug_trace(None, 0)
    t = buf.cpu().numpy()
    if args.raw:
        for li in range(args.launches):
            g0 = t[li, 0]
            if g0[6] > 0 and g0[9] > 0 and g0[5] > g0[0] and g0[10] == 0:       # a gemm_tc launch (globaltimer ns)
                print(f"launch {li} gemm_tc mtiles {g0[6]} K {g0[7]} N {g0[8]} bn {g0[9]}: prologue {g0[1]-g0[0]} ns, "
                      f"pdl wait {g0[2]-g0[1]}, k loop {g0[3]-g0[2]}, epilogue {g0[4]-g0[3]}, tail {g0[5]-g0[4]}")
                continue
            for role in range(3):
                w = t[li, role]
                n = int((w != 0).sum())
                if n > 1:
                    if role == 0:
                        g = t[li, 3]
                        if g[0]:
                            print(f"launch {li} globaltimer ns: cta0 entry->sync {g[1]-g[0]} sync->pdl {g[2]-g[1]} pdl->exit {g[3]-g[2]}; "
                                  f"last cta: entry(rel cta0) {g[8]-g[0]} entry->sync {g[9]-g[8]} sync->pdl {g[10]-g[9]} pdl->exit {g[11]-g[10]}")
                    print(f"launch {li} role {role}: {n} stamps, span {(w[n - 1] - w[0]) / 1.9e3:.1f} us; deltas",
                          [int(w[i + 1] - w[i]) for i in range(n - 1)])
        return
    for li in range(args.launches):
        w0, w1, mm = t[li, 0], t[li, 1], t[li, 2]
        n0 = int((w0 != 0).sum())
        if n0 == 0:
            continue
        base = min(x for x in (w0[0], w1[0] if w1[0] else w0[0], mm[0] if mm[0] else w0[0]))
        print(f"--- tile launch {li}: worker0 {n0} stamps, worker1 {int((w1 != 0).sum())}, mma {int((mm != 0).sum())}; "
              f"span {(max(w0.max(), w1.max()) - base) / 1.9e3:.1f} us (cycles / 1.9 GHz)")
        for name, w in (("w0", w0), ("w1", w1)):
            n = int((w != 0).sum())
            rows = []
            for i in range(0, n - 2, 3):
                e0, e1, e2 = w[i], w[i + 1], w[i + 2]
                prev = w[i - 1] if i else base
                rows.append(f"[{(e0 - base) / 1.9e3:6.1f}us pre {(e0 - prev):6d} wait {(e1 - e0):6d} epi {(e2 - e1):6d}]")
            print(name, " ".join(rows))
        n = int((mm != 0).sum())
        print("mma", " ".join(f"[{(mm[i] - base) / 1.9e3:6.1f}us issue {(mm[i + 1] - mm[i]):5d}]" for i in range(0, n - 1, 2)))


if __name__ == "__main__":
    main()
