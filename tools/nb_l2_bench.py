#!/usr/bin/env python
"""Cost of the L2-ball update against the L-inf one inside whole NB attacks (TF32 mode, SSG, random-init weights).

Two workloads, each run with norm="Linf" and norm="L2", alternating, 7 timed attacks per arm after one warm-up attack:
  * config 2 of BASELINE.json: tar_NB_attack, B = 16 x 4096, 50 iterations, target 7 on the class-11 points;
  * NB_attack (non-targeted), B = 16 x 4096, 50 iterations.
An attack is timed with CUDA events around the whole call (geometry pass included); steps/s = iterations / time.  The
PF_PGD family ("pgd_update": the update kernels) is then read per step from the library's event profiler in a separate
run.  The card's name and power limit are read in the same process.  Writes one JSON file (``--out``)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointsecguard_b200 import _lib as L, synthetic as syn, torchattacks  # noqa: E402
from pointsecguard_b200.engine import MLP_TF32  # noqa: E402
from pointsecguard_b200.models.pointnet2_sem_seg import get_model  # noqa: E402

B, N, ITERS, REPS = 16, 4096, 50, 7
TARGET, ORIGIN = 7, 11
# (eps, alpha): the bench's L-inf values; for L2 a ball of radius 2 in the colour space of a block's moving points
PARAMS = {"Linf": (0.5, 0.1), "L2": (2.0, 0.25)}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True, check=True).stdout
    name, power, clk = [s.strip() for s in out.strip().split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def pgd_ms_per_step(run):
    L.psg_prof_enable(1)
    torch.manual_seed(0)
    run()
    torch.cuda.synchronize()
    n = L.psg_prof_ncat()
    ms, cnt = (C.c_double * n)(), (C.c_int64 * n)()
    L.psg_prof_collect(ms, cnt)
    L.psg_prof_enable(0)
    fam = {L.psg_prof_name(i).decode(): (ms[i], cnt[i]) for i in range(n)}
    t, c = fam["pgd_update"]
    return {"pgd_update_ms_per_step": t / ITERS, "pgd_update_launches": int(c),
            "all_families_ms_per_step": sum(v[0] for v in fam.values()) / ITERS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles",
                                                  "nb_l2_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nb_l2_bench needs a CUDA device")
    info = gpu_info()
    model = get_model(13)
    model.load_state_dict(syn.make_state_dict("ssg", init="he"))
    model = model.cuda().eval()
    model.set_mlp_mode(MLP_TF32)
    x, labels = syn.make_painted_blocks(B, N, 0)
    xd, lab = x.cuda(), labels.numpy().astype(np.float64)
    mask = (labels == ORIGIN).numpy()

    def attack(workload, norm):
        eps, alpha = PARAMS[norm]
        if workload == "tar_nb":
            atk = torchattacks.tar_NB_attack(model, eps=eps, alpha=alpha, iters=ITERS, target=TARGET, mask=mask, norm=norm)
        else:
            atk = torchattacks.NB_attack(model, eps=eps, alpha=alpha, iters=ITERS, norm=norm)
        return lambda: atk(xd, lab)

    result = {"tool": "tools/nb_l2_bench.py", **info, "mlp_mode": "tf32", "B": B, "N": N, "iterations": ITERS,
              "timed_attacks_per_arm": REPS, "params": PARAMS, "workloads": {}}
    for workload in ("tar_nb", "nb"):
        runs = {norm: attack(workload, norm) for norm in PARAMS}
        for run in runs.values():                                     # warm-up: one whole attack per arm
            torch.manual_seed(0)
            run()
        torch.cuda.synchronize()
        ms = {norm: [] for norm in PARAMS}
        for _ in range(REPS):
            for norm, run in runs.items():                            # alternating arms
                torch.manual_seed(0)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run()
                e1.record()
                e1.synchronize()
                ms[norm].append(e0.elapsed_time(e1))
        arms = {}
        for norm, run in runs.items():
            t = np.array(ms[norm])
            arms[norm] = {"attack_ms_median": float(np.median(t)), "attack_ms_min": float(t.min()),
                          "attack_ms_max": float(t.max()), "steps_per_s_median": ITERS * 1e3 / float(np.median(t)),
                          "steps_per_s_min": ITERS * 1e3 / float(t.max()), "steps_per_s_max": ITERS * 1e3 / float(t.min()),
                          **pgd_ms_per_step(run)}
        result["workloads"][workload] = arms
        print(workload, json.dumps(arms), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "power_limit", "max_sm_clock")}))


if __name__ == "__main__":
    main()
