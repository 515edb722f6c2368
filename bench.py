#!/usr/bin/env python
"""bench.py -- PGD attack steps/sec on 4096-pt PointNet++ sem-seg blocks (BASELINE.json metric).

A *step* is one PGD iteration (one forward + one input-gradient backward + the fused perturbation
update) for a batch of 16 S3DIS-shaped 4096-point blocks per GPU: BASELINE.json configs[1]
(PointNet++ SSG sem-seg, norm-bounded targeted PGD, B=16x4096, random-init weights, synthetic data).
One timed region is one ``tar_NB_attack(iters=K)`` call -- EXACTLY K steps: the batched geometry pass
(FPS, ball query, 3-NN, CSRs for all K forwards), the FPS start draws on the CPU generator, and the
K-step loop.  The region is repeated ``--repeats`` times (L2 flushed before each); ``value`` is the
median (min / max reported), each repeat the max over ranks.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); every rank attacks its own 16 blocks (weak
scaling, no data-path collective) and the per-class counters are all-reduced over NCCL afterwards.
``--impl reference`` times the UNMODIFIED reference (its own ``torchattacks.tar_NB_attack`` over its
own ``pointnet2_sem_seg.get_model``, imported from oracle/_ref, see oracle/build_ref.py) on the host
cores at the full B=16; if oracle/_ref is absent it falls back to the oracle port and says so.
``--dump-outputs DIR`` writes what the last timed attack returned as ``DIR/adv.npy`` (float32 [B,9,N], the global batch
in rank order): the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

B_PER_GPU = 16
N_POINTS = 4096
EPS, ALPHA, TARGET, ORIGIN = 0.5, 0.1, 7, 11          # NB_target_test_semseg.py:177, :48-49
FLOPS_PER_BLOCK_STEP = 3.880e9                        # SURVEY.md App. C: forward + dgrad, SSG, N=4096
MSG_FLOPS_PER_BLOCK_STEP = 6.098e9
METRIC = "pgd_attack_steps_per_sec"
UNIT = "steps/s (1 step = fwd + input-grad bwd + update of 16 blocks x 4096 pts per GPU)"


def config_dict():
    """The workload both arms run (identical dict in both JSON lines)."""
    return {"workload": "configs[1]: PointNet++ SSG sem_seg, norm-bounded targeted PGD (tar_NB_attack eps=0.5 alpha=0.1 "
                        "target=7, mask=class 11), B=16x4096 per GPU, random-init weights, synthetic S3DIS-shaped blocks",
            "blocks_per_gpu": B_PER_GPU, "points": N_POINTS, "channels": 9, "classes": 13,
            "weights": "random-init (synthetic.make_state_dict('ssg', init='he'))",
            "inputs": "synthetic.make_painted_blocks(16 x n_gpus, 4096, seed 0)"}


def peaks():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML)."""
    BAD = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown"}
    NOTE = {0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.maxclk = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.maxclk = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in {**self.BAD, **self.NOTE}.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.01)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.maxclk, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.maxclk, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# stdout carries exactly ONE JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its
# version banner there at any NCCL_DEBUG level from VERSION up, whatever NCCL_DEBUG_FILE says), so main() points fd 1 at
# stderr for the whole run and the line goes out through a private duplicate of the original stdout.
_JSON_FD = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def dump_outputs(out_dir, arrays):
    """Writes each array of ``arrays`` as ``out_dir/<name>.npy`` in float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def make_inputs(B, seed=0):
    from pointsecguard_b200 import synthetic as syn
    x, labels = syn.make_painted_blocks(B, N_POINTS, seed)
    mask = labels == ORIGIN                                  # per-block masks, [B,N]
    return x, labels, mask


# --------------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference from oracle/_ref (fallback: the oracle port)
# --------------------------------------------------------------------------------------------------
def cpu_reference(steps, warmup_steps):
    """Times ``steps`` iterations of the reference's own tar_NB_attack on the full 16-block batch on all host threads,
    after one warm-up attack of ``warmup_steps`` iterations.  Returns (steps/s, cores, kind, sample string, seconds,
    the timed attack's perturbed blocks).

    The reference class handles a batch by reading ``labels[0]`` / ``outputs[0]`` (target.py:26,36): it runs the forward
    and the backward of all 16 blocks (the full cost of a 16-block step) with a [N] mask, which is what is timed; per-block
    masks do not exist in the reference."""
    from pointsecguard_b200 import synthetic as syn
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    x, labels, mask = make_inputs(B_PER_GPU, 0)
    sd = syn.make_state_dict("ssg", init="he")
    lab_np = labels.numpy().astype(np.float64)
    try:
        from oracle import build_ref
        ssg, _, ta = build_ref.import_reference()
        model = ssg.get_model(13)
        model.load_state_dict(sd)
        model = model.eval()
        mk = lambda it: ta.tar_NB_attack(model, eps=EPS, alpha=ALPHA, iters=it, target=TARGET, mask=mask[0].numpy())
        run = lambda it: mk(it)(x, lab_np)
        kind, who = "reference", "unmodified reference from oracle/_ref (torchattacks.tar_NB_attack on pointnet2_sem_seg.get_model)"
    except ImportError as e:
        from oracle import attacks_oracle as AO
        from oracle import pointnet2_oracle as PO
        PO.GEOMETRY = "torch"          # op-for-op the reference's geometry (Python FPS loop, matmul + sort)
        model = PO.OracleModel(sd, "ssg")
        run = lambda it: AO.tar_nb_attack(model, x, lab_np, eps=EPS, alpha=ALPHA, iters=it, target=TARGET, mask=mask)
        kind, who = "port", f"oracle port with the reference's op-for-op geometry (oracle/_ref unavailable: {e})"
    torch.manual_seed(0)
    if warmup_steps > 0:
        run(warmup_steps)
    t0 = time.perf_counter()
    adv = run(steps)
    dt = time.perf_counter() - t0
    sps = steps / dt
    sample = (f"tar-NB SSG, all 16 blocks x {steps} iterations (+ a warm-up attack of {warmup_steps}) on {cores} threads, "
              f"{dt:.1f} s; {who}")
    return sps, cores, kind, sample, dt, adv


def run_reference(args, rank):
    if rank != 0:
        return
    sps, cores, kind, sample, dt, adv = cpu_reference(args.steps, max(0, min(args.warmup, 5)))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"adv": adv.detach().numpy()})
    line = {
        "impl": "reference", "metric": METRIC, "value": sps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 / sps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(),
        "timed_steps": args.steps, "timed_seconds": dt,
        "cpu_baseline": {"value": sps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": sps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
def _flops_rows_chain(widths):
    """forward FLOPs per row of a conv chain [c0 -> c1 -> ...]"""
    return sum(2 * a * b for a, b in zip(widths[:-1], widths[1:]))


def measure_tf32_peak(dev, seconds=1.5):
    """Dense TF32 tensor-core rate measured the way MEASURED_PEAKS.json measured bf16: torch.matmul 8192^3 (cuBLAS) with
    TF32 allowed; best of 10 (burst) and back to back for ``seconds`` (sustained).  Runs AFTER the timed regions."""
    n = 8192
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        for _ in range(3):
            torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        fl = 2.0 * n ** 3
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch.matmul(a, b, out=c); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(10, int(seconds * 1e3 / best))
        e0.record()
        for _ in range(reps):
            torch.matmul(a, b, out=c)
        e1.record(); torch.cuda.synchronize()
        sus = e0.elapsed_time(e1) / reps
        return {"burst_tflops": fl / (best / 1e3) / 1e12, "sustained_tflops": fl / (sus / 1e3) / 1e12,
                "how": f"torch.matmul fp32 8192^3 with allow_tf32 (cuBLAS): best of 10 / {reps} back to back"}
    except Exception as e:          # never lose the bench line to the peak probe
        return {"burst_tflops": None, "sustained_tflops": None, "how": f"failed: {e}"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def run_native(args, rank, world, local_rank):
    import ctypes as C
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from pointsecguard_b200 import _lib as L
    from pointsecguard_b200 import distributed as D
    from pointsecguard_b200 import synthetic as syn, torchattacks
    from pointsecguard_b200 import metrics as MT
    from pointsecguard_b200.engine import MLP_FP32, MLP_TF32
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model

    for opt in ("sa_ng", "clusters", "fp_min_tiles", "fp_slabs", "ts", "deep", "segsum_warp", "sa_grid_div"):                 # A/B switches of the library (experiments only)
        if os.environ.get("PSG_OPT_" + opt.upper()):
            L.psg_set_option(opt.encode(), int(os.environ["PSG_OPT_" + opt.upper()]))
    model = get_model(13)
    model.load_state_dict(syn.make_state_dict("ssg", init="he"))      # the configuration's random-init network
    model = model.to(dev).eval()
    mode = MLP_TF32 if args.mlp == "tf32" else MLP_FP32
    model.set_mlp_mode(mode)
    # weak scaling: a global batch of 16 blocks per GPU; every rank builds the same global batch from
    # the seed, keeps its contiguous slice, and draws FPS starts for the GLOBAL batch (sliced), so an
    # N-GPU run attacks exactly the blocks a 1-GPU run of the same global batch would, with the same draws
    shard = D.shard_for(B_PER_GPU * world, rank, world)
    model.set_shard(shard if world > 1 else None)
    x_all, labels_all, mask_all = make_inputs(B_PER_GPU * world, seed=0)
    x_host, labels, mask = shard.slice(x_all), shard.slice(labels_all), shard.slice(mask_all)
    x_pin = x_host.contiguous().pin_memory()                      # [B,9,N] contiguous pinned host copy
    x_dev = x_host.to(dev)
    adv_host = torch.empty(x_pin.shape, dtype=torch.float32).pin_memory()      # e2e: the perturbed blocks land here
    lab_np = labels.numpy().astype(np.float64)
    K, W, R = args.steps, args.warmup, max(1, args.repeats)
    mk = lambda iters: torchattacks.tar_NB_attack(model, eps=EPS, alpha=ALPHA, iters=iters, target=TARGET, mask=mask)
    atk = mk(K)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)    # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms_list):
        t = torch.tensor(ms_list, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.cpu().numpy()

    # warm-up: W untimed steps, then one untimed attack at the timed geometry-chunk size
    if W > 0:
        mk(W)(x_dev, lab_np)
    mk(min(K, 64))(x_dev, lab_np)

    # ---- device-resident timing: R repeats of EXACTLY K steps, inputs already in HBM ----
    # clocks are sampled on rank 0 only (its line carries them; eight ranks polling NVML at once stalled each other's
    # first launches), and the sampler thread is already running when the first timed region starts
    clocks = ClockSampler(local_rank) if rank == 0 else None
    if clocks is not None:
        clocks.start()
        time.sleep(0.03)
    # resident and end-to-end repeats ALTERNATE, so both medians see the same clocks, straggler ranks and thermal state (timed
    # one block after the other, the noise between the blocks exceeded the copy cost the end-to-end number adds)
    ms_res, ms_e2e, launches, adv, wall = [], [], 0, None, 0.0
    for r in range(R):
        # ---- inputs already in HBM ----
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.manual_seed(0)
        flush.fill_(r & 0xFF)
        barrier()
        l0 = L.psg_launch_count()
        e0.record()
        adv = atk(x_dev, lab_np)
        e1.record()
        barrier()
        launches = L.psg_launch_count() - l0
        ms_res.append(e0.elapsed_time(e1))
        # ---- end to end through the public API from pinned host memory, result read back ----
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.manual_seed(0)
        flush.fill_((r + 101) & 0xFF)
        barrier()
        t0 = time.perf_counter()
        e0.record()
        xd = x_pin.to(dev, non_blocking=True)
        adv2 = atk(xd, lab_np)
        adv_host.copy_(adv2, non_blocking=True)          # result read back into pinned host memory
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms_e2e.append(e0.elapsed_time(e1))
    ms_res = max_over_ranks(ms_res)
    ms_total = float(np.median(ms_res))
    value = world * K / (ms_total / 1e3)
    clk = clocks.finish() if clocks is not None else None
    ms_e2e = max_over_ranks(ms_e2e)
    e2e_ms = float(np.median(ms_e2e))
    e2e_value = world * K / (e2e_ms / 1e3)
    h2d = x_pin.numel() * 4 / K
    d2h = adv_host.numel() * 4 / K
    same_as_resident = bool(torch.equal(adv_host, adv.cpu()))
    if args.dump_outputs:
        out = adv.contiguous()
        if world > 1:
            full = torch.empty((world * out.shape[0],) + tuple(out.shape[1:]), dtype=out.dtype, device=dev)
            dist.all_gather_into_tensor(full, out)
            out = full
        if rank == 0:
            dump_outputs(args.dump_outputs, {"adv": out.cpu().numpy()})

    # ---- metrics + the only collective: per-class counters all-reduced over NCCL (timed on its own) ----
    torch.manual_seed(1)
    logp_adv, _ = model(adv)
    counters = MT.attack_counters(logp_adv, labels.to(dev), mask.to(dev), TARGET)
    barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    D.all_reduce_sum_(counters)
    a1.record()
    torch.cuda.synchronize()
    allreduce_us = float(max_over_ranks([a0.elapsed_time(a1) * 1e3])[0]) if world > 1 else 0.0
    summary = MT.summarize(counters.cpu(), 13)

    # ---- N > 1: BASELINE configs[3] -- MSG, a GLOBAL batch of 64 blocks sharded over the ranks, counters all-reduced ----
    config4 = run_config4_msg(args, rank, world, dev, barrier, max_over_ranks) if world > 1 else None

    line = None
    if rank == 0:
        model.set_shard(None)
        # ---- live per-kernel-family timing (CUDA event pairs on the launching stream) ----
        L.psg_prof_enable(1)
        torch.manual_seed(0)
        mk(K)(x_dev, lab_np)          # same attack length as the timed run: the batched geometry pass amortises alike
        ncat = L.psg_prof_ncat()
        msb = (C.c_double * ncat)()
        cnt = (C.c_int64 * ncat)()
        L.psg_prof_collect(msb, cnt)
        L.psg_prof_enable(0)
        fam = {L.psg_prof_name(i).decode(): {"ms_per_step": msb[i] / K, "launches_per_step": cnt[i] / K}
               for i in range(ncat) if cnt[i]}
        pk = peaks()
        tf32 = measure_tf32_peak(dev)
        if args.mlp == "tf32" and tf32["sustained_tflops"]:
            peak, peak_src = tf32["sustained_tflops"], "TF32 measured in this run (sustained, " + tf32["how"] + ")"
        else:
            peak, peak_src = pk["bf16_tflops_sustained"] / 2.0, pk["source"] + " bf16 sustained / 2"
        rows0 = B_PER_GPU * N_POINTS
        step_flops = FLOPS_PER_BLOCK_STEP * B_PER_GPU
        # dominant FAMILY by time; the roofline object describes its launches
        mlp_fams = ("sa_fused_fwd", "sa_fused_bwd", "fp_fused_fwd", "fp_fused_bwd", "head_chain", "gemm_fwd", "gemm_bwd")
        dom_name = max((k for k in fam if k in mlp_fams), key=lambda k: fam[k]["ms_per_step"], default=None)
        fam_flops = family_flops()
        if dom_name is not None:
            dom = fam[dom_name]
            fl = fam_flops.get(dom_name, 0.0) * B_PER_GPU
            ach = fl / (dom["ms_per_step"] / 1e3) / 1e12 if dom["ms_per_step"] else 0.0
            roofline = {"bound": "tensor", "kernel": f"{dom_name} (the kernel family with the largest share of the step, "
                                                     f"{dom['launches_per_step']:.0f} launches/step)",
                        "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_source": peak_src,
                        "flops_per_step_in_family": fl, "ms_per_step_in_family": dom["ms_per_step"],
                        "traffic": _ncu_traffic(dom_name),
                        "traffic_note": "DRAM bytes per launch from the committed cold-cache `ncu --set full` capture "
                                        "(profiles/ncu_traffic.json), not measured in this run"}
        else:
            roofline = {"bound": "tensor", "kernel": None, "achieved": 0.0, "peak": peak, "unit": "TFLOP/s", "frac": 0.0,
                        "traffic": None, "peak_source": peak_src}
        roofline["step"] = {"tflops": value / world * step_flops / 1e12, "frac": value / world * step_flops / 1e12 / peak,
                            "flops_per_step": step_flops,
                            "note": "whole step incl. geometry, gathers, segmented sums and update: algorithmic MLP FLOPs "
                                    "(forward + dgrad, SURVEY App. C) / measured step time"}
        roofline["families"] = {k: {"ms_per_step": round(fam[k]["ms_per_step"], 4),
                                    "tflops": fam_flops[k] * B_PER_GPU / (fam[k]["ms_per_step"] / 1e3) / 1e12,
                                    "frac": fam_flops[k] * B_PER_GPU / (fam[k]["ms_per_step"] / 1e3) / 1e12 / peak}
                                for k in fam if k in fam_flops and fam[k]["ms_per_step"] > 0}
        roofline["tf32_peak_measured"] = tf32
        roofline["mlp_mode"] = args.mlp
        # HBM-side primitives (SURVEY.md 8d byte formulas, all four levels), achieved GB/s vs measured copy bandwidth
        npts = [N_POINTS, 1024, 256, 64, 16]
        byt = {"fps": sum(12 * npts[l] + 8 * npts[l + 1] for l in range(4)),
               "ball_query": sum(12 * npts[l] + 12 * npts[l + 1] + 8 * npts[l + 1] * 32 for l in range(4)),
               "three_nn": sum(12 * npts[l] + 12 * npts[l + 1] + 36 * npts[l] for l in range(4))}
        roofline["primitives_hbm"] = {
            k: {"GBps": byt[k] * B_PER_GPU / (fam[k]["ms_per_step"] / 1e3) / 1e9,
                "frac_of_hbm": byt[k] * B_PER_GPU / (fam[k]["ms_per_step"] / 1e3) / 1e9 / pk["hbm_gbs"]}
            for k in byt if k in fam}
        # ---- the same workload in the two parity-grade modes (rtol 1e-3 against the reference): 3xTF32 on tcgen05
        # (error-compensated per-layer GEMMs) and the CUDA-core fp32 GEMMs ----
        parity = None
        if args.mlp == "tf32" and not args.no_parity:
            from pointsecguard_b200.engine import MLP_TF32X3
            legs = {}
            for name, pm in (("tf32x3", MLP_TF32X3), ("fp32", MLP_FP32)):
                model.set_mlp_mode(pm)
                for _ in range(2):                     # full-length warm-up attacks: a short one would not bind the second
                    mk(K)(x_dev, lab_np)               # engine of the geometry head start or pick the kernels' tile counts
                ms_p = []
                for r in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.manual_seed(0)
                    flush.fill_(r)
                    torch.cuda.synchronize()
                    e0.record(); adv_p = mk(K)(x_dev, lab_np); e1.record()
                    torch.cuda.synchronize()
                    ms_p.append(e0.elapsed_time(e1))
                msp = float(np.median(ms_p))
                if os.environ.get("PSG_BENCH_DEBUG"):
                    print(f"parity leg {name}: ms per attack {ms_p}", file=sys.stderr)
                st_t, st_p = (np.rint(((a[:, 3:6] - x_dev[:, 3:6]) / ALPHA).cpu().numpy()) for a in (adv, adv_p))
                mk3 = mask.unsqueeze(1).expand(-1, 3, -1).numpy()
                legs[name] = {"value": K / (msp / 1e3), "ms_per_step": msp / K,
                              "tf32_identical_steps_on_masked_points": float((st_t[mk3] == st_p[mk3]).mean())}
            model.set_mlp_mode(mode)
            parity = {"mlp": "tf32x3", "value": legs["tf32x3"]["value"], "unit": UNIT, "ms_per_step": legs["tf32x3"]["ms_per_step"],
                      "what": "tcgen05 with the 3xTF32 split (A_lo W_hi + A_hi W_lo + A_hi W_hi; fused SA1 / SA2 and fp1 + head kernels, "
                              "per-layer GEMMs elsewhere): the fp32 gates of tests/test_gpu_model.py / test_gpu_configs.py hold "
                              "(logits rtol 1e-3, gradient rel < 1e-4, last-step replay >= 99.5 %)",
                      "fp32_cuda_cores": legs["fp32"], "tf32x3": legs["tf32x3"]}
        # ---- attack quality on the TRAINED synthetic checkpoint, against the oracle's golden run of the same call ----
        quality = attack_quality(dev, mode)
        # ---- CPU baseline (bounded sample of the same workload on the host cores) ----
        if args.no_cpu or world > 1:          # the CPU leg runs on rank 0 at N = 1 only
            cpu = None
        else:
            sps, cores, kind, sample, _, _ = cpu_reference(5, 1)
            cpu = {"value": sps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.mlp == "fp32" else "tf32", "data": "synthetic", "config": config_dict(),
            "timing": {"repeats": R, "statistic": "median over repeats of (max over ranks)", "steps_per_repeat": K,
                       "ms_per_attack": {"median": ms_total, "min": float(ms_res.min()), "max": float(ms_res.max())},
                       "value_min": world * K / (float(ms_res.max()) / 1e3), "value_max": world * K / (float(ms_res.min()) / 1e3),
                       "l2": "256 MB buffer written before each timed attack (L2 flush); steps inside an attack run back to "
                             "back as in the reference loop"},
            "tolerance": "fp32 and 3xTF32 modes (parity_mode): logits rtol 1e-3, colour-gradient rel < 1e-4 (measured 3.4e-6 / 4.5e-6), "
                         "last-step replay >= 99.5 % identical (measured 99.98 %+); tf32 mode (timed): |dlogp| < 5e-3, "
                         "colour-gradient rel < 8e-2, sign > 99 % vs the REFERENCE goldens, acc / mIoU / target hit-rate within "
                         "0.5 pt of the oracle at B=16 x 50 iterations (tests/test_gpu_configs.py); FPS / ball-query / 3-NN "
                         "indices bit-exact in every mode",
            "block_steps_per_s": value * B_PER_GPU,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_attack": {"median": e2e_ms, "min": float(ms_e2e.min()), "max": float(ms_e2e.max())},
                    "wall_s_last_repeat": wall, "identical_to_resident_run": same_as_resident},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": roofline,
            "kernel_families_ms_per_step": {k: round(v["ms_per_step"], 4) for k, v in fam.items()},
            "kernel_families_note": "event pairs around each launch; consecutive launches overlap under programmatic dependent "
                                    "launch, so per-family times are upper bounds and sum to more than ms_per_step",
            "parity_mode": parity,
            "cpu_baseline": cpu,
            "attack_metrics": summary,
            "attack_metrics_note": "random-init network of the timed configuration (uninformative by construction); see attack_quality",
            "attack_quality": quality,
            "counter_allreduce_us": allreduce_us,
        }
        if config4 is not None:
            line["config4_msg"] = config4
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def family_flops():
    """Algorithmic FLOPs per block-step of the SSG network by kernel family (forward or dgrad of the layers each family
    runs in tcgen05 mode; SURVEY.md App. C shapes)."""
    sa = lambda rows, w: rows * _flops_rows_chain(w)
    sa12 = sa(1024 * 32, [12, 32, 32, 64]) + sa(256 * 32, [67, 64, 64, 128])
    sa34 = sa(64 * 32, [131, 128, 128, 256]) + sa(16 * 32, [259, 256, 256, 512])
    fp234 = 64 * _flops_rows_chain([768, 256, 256]) + 256 * _flops_rows_chain([384, 256, 256]) + 1024 * _flops_rows_chain([320, 256, 128])
    head = 4096 * _flops_rows_chain([128, 128, 128, 128, 128, 13])
    return {"sa_fused_fwd": sa12 + sa34, "sa_fused_bwd": sa12 + sa34, "fp_fused_fwd": fp234, "fp_fused_bwd": fp234,
            "head_chain": 2 * head}


def attack_quality(dev, mode):
    """The timed attack on the trained painted-blocks checkpoint (one GPU, 16 blocks, 50 iterations): clean / adversarial
    acc, mIoU and target hit-rate next to the oracle's golden run of the same call (tests/golden/atsize_config2.npz)."""
    try:
        from pointsecguard_b200 import metrics as MT
        from pointsecguard_b200 import synthetic as syn, torchattacks
        from pointsecguard_b200.models.pointnet2_sem_seg import get_model
        m = get_model(13)
        m.load_state_dict(syn.load_checkpoint("ssg"))
        m = m.to(dev).eval()
        m.set_mlp_mode(mode)
        x, labels, mask = make_inputs(B_PER_GPU, 0)
        xd = x.to(dev)

        def met(t):
            torch.manual_seed(1)
            return MT.summarize(MT.attack_counters(m(t)[0], labels.to(dev), mask.to(dev), TARGET).cpu(), 13)
        clean = met(xd)
        torch.manual_seed(0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        adv = torchattacks.tar_NB_attack(m, eps=EPS, alpha=ALPHA, iters=50, target=TARGET, mask=mask)(xd, labels.numpy().astype(np.float64))
        e1.record()
        after = met(adv)
        out = {"checkpoint": "tests/golden/ckpt_ssg_painted.npz (300 Adam steps on synthetic painted blocks)", "iterations": 50,
               "clean": {k: clean[k] for k in ("acc", "miou", "target_acc")},
               "adversarial": {k: after[k] for k in ("acc", "miou", "target_acc")},
               "steps_per_s": 50 / (e0.elapsed_time(e1) / 1e3)}
        g = np.load(os.path.join(REPO, "tests", "golden", "atsize_config2.npz"))
        out["oracle"] = {k: float(g["adv_" + k]) for k in ("acc", "miou", "target_acc")}
        out["within_half_point_of_oracle"] = bool(all(abs(after[k] - out["oracle"][k]) < 0.005 for k in ("acc", "miou", "target_acc")))
        st = np.rint(((adv[:, 3:6] - xd[:, 3:6]) / ALPHA).cpu().numpy()).astype(np.int8)
        mk3 = mask.unsqueeze(1).expand(-1, 3, -1).numpy()
        out["identical_step_counts_on_masked_points"] = float((st[mk3] == g["steps"][mk3]).mean())
        return out
    except Exception as e:
        return {"error": repr(e)}


def run_config4_msg(args, rank, world, dev, barrier, max_over_ranks):
    """BASELINE configs[3]: MSG sem-seg, a global batch of 64 blocks sharded over the ranks (32 / 16 / 8 per GPU), NB_attack
    10 iterations, per-class counters all-reduced; rank 0 re-runs the whole batch alone and compares the counters."""
    try:
        import torch.distributed as dist
        from pointsecguard_b200 import distributed as D
        from pointsecguard_b200 import metrics as MT
        from pointsecguard_b200 import synthetic as syn, torchattacks
        from pointsecguard_b200.engine import MLP_TF32
        from pointsecguard_b200.models.pointnet2_sem_seg_msg import get_model
        G, IT = 64, 10
        m = get_model(13)
        m.load_state_dict(syn.load_checkpoint("msg"))
        m = m.to(dev).eval()
        m.set_mlp_mode(MLP_TF32)
        x, labels = syn.make_painted_blocks(G, N_POINTS, 0)
        sh = D.shard_for(G, rank, world)
        m.set_shard(sh)
        xs, ls = sh.slice(x).to(dev), sh.slice(labels)
        lab_np = ls.numpy().astype(np.float64)
        atk = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=IT)
        atk(xs, lab_np)
        ms, adv = [], None
        for r in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.manual_seed(0)
            barrier()
            e0.record(); adv = atk(xs, lab_np); e1.record()
            barrier()
            ms.append(e0.elapsed_time(e1))
        ms = float(np.median(max_over_ranks(ms)))
        torch.manual_seed(1)
        cnt = MT.attack_counters(m(adv)[0], ls.to(dev))
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(); D.all_reduce_sum_(cnt); a1.record()
        torch.cuda.synchronize()
        ar_us = float(max_over_ranks([a0.elapsed_time(a1) * 1e3])[0])
        out = {"workload": f"MSG sem_seg, NB_attack eps=0.1 alpha=0.05 x {IT} iterations, global batch {G} sharded over {world} GPUs "
                           f"({G // world} blocks per GPU), trained painted-blocks checkpoint", "scaling": "strong",
               "steps_per_s": IT / (ms / 1e3), "ms_per_step": ms / IT, "allreduce_us": ar_us,
               "adv": {k: v for k, v in MT.summarize(cnt.cpu(), 13).items() if k in ("acc", "miou", "points")}}
        if rank == 0:
            # single-GPU run of the same global batch with the same draws: the counters must be equal exactly
            import pointsecguard_b200.distributed as DD
            ws = DD.world_size
            DD.world_size = lambda: 1
            m.set_shard(None)
            try:
                atk1 = torchattacks.NB_attack(m, eps=0.1, alpha=0.05, iters=IT)
                atk1(x.to(dev), labels.numpy().astype(np.float64))
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.manual_seed(0)
                torch.cuda.synchronize()
                e0.record(); adv1 = atk1(x.to(dev), labels.numpy().astype(np.float64)); e1.record()
                torch.cuda.synchronize()
                torch.manual_seed(1)
                c1 = MT.attack_counters(m(adv1)[0], labels.to(dev))
                out["counters_equal_single_gpu"] = bool(torch.equal(c1, cnt))
                out["single_gpu_steps_per_s"] = IT / (e0.elapsed_time(e1) / 1e3)
            finally:
                DD.world_size = ws
        dist.barrier()
        return out
    except Exception as e:
        return {"error": repr(e)}


def _ncu_traffic(kernel):
    """dram bytes (read + write) per launch of `kernel` from the committed ncu --set full summary, or None."""
    try:
        with open(os.path.join(REPO, "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=7, help="timed attacks of --steps steps each (median reported)")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--mlp", default=os.environ.get("PSG_MLP", "tf32"), choices=["fp32", "tf32"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the fp32 parity-mode leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the perturbed blocks of the last timed attack to DIR/adv.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun for --gpus > 1")
    run_native(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
