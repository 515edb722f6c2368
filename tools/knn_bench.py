"""Time the dense kNN graph (csrc/knn.cu) at ResGCN-28's sizes against the reference's own ops on the same GPU.

One ResGCN-28 forward builds 28 graphs on N = 4096 points: the head's on xyz (C = 3, k = 16) and one per backbone block i on its
64-wide feature map (k * dilation = 16 * (1 + i), i = 0 ... 26).  Each is timed with CUDA events after warm-up, through
``psg_dense_knn`` and through the reference's ops (``-2 x x^T`` by matmul with TF32 off, the two squared norms, then
``torch.topk``).  The inputs (0.2 MB per cloud at C = 3, 1 MB at C = 64) stay resident in the 126 MB L2 across repetitions,
as they do inside a forward.  Also timed: both kernels around their boundary, the register kernel at k = 16 and the
shared-memory list kernel at k = 17, 32 and 33 (it serves k > 16 at C <= 64).  Prints one JSON document and writes it to --out.

    python tools/knn_bench.py --out /tmp/knn_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointsecguard_b200 import _lib as L  # noqa: E402

N = 4096
RESGCN_K, RESGCN_BLOCKS = 16, 27


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True, check=True).stdout
    name, power, clk = [s.strip() for s in out.strip().split(",")]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    mhz = float(clk.split()[0])
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk, "sms": sms,
            "fp32_fma_peak_tflops": 2 * 128 * sms * mhz * 1e6 / 1e12}


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def ours(x, k, out):
    B, n, C = x.shape
    st = torch.cuda.current_stream().cuda_stream
    return lambda: L.psg_dense_knn(x.data_ptr(), B, n, C, k, out.data_ptr(), None, st)


def reference(x, k):
    def f():
        inner = -2 * torch.matmul(x, x.transpose(2, 1))
        sq = torch.sum(torch.mul(x, x), dim=-1, keepdim=True)
        return torch.topk(-(sq + inner + sq.transpose(2, 1)), k=k)[1]
    return f


def forward_calls(B, g):
    xyz = torch.rand(B, N, 3, generator=g).cuda()
    feat = torch.randn(B, N, 64, generator=g).cuda()
    return [("head", xyz, RESGCN_K)] + [(f"block{i}", feat, RESGCN_K * (1 + i)) for i in range(RESGCN_BLOCKS)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    info = gpu_info()
    res = {"info": info, "note": "inputs are L2-resident (a few MB); times are CUDA-event means after warm-up",
           "forward": {}, "boundary": {}}
    g = torch.Generator().manual_seed(0)
    for B in (16, 1):
        rows = []
        for name, x, k in forward_calls(B, g):
            out = torch.empty(B, N, k, dtype=torch.int64, device="cuda")
            t = timed(ours(x, k, out), a.warmup, a.reps)
            tr = timed(reference(x, k), a.warmup, a.reps)
            pairs = B * N * N
            flop = pairs * 2 * x.shape[-1]
            rows.append({"call": name, "C": x.shape[-1], "k": k, "ms": t, "ref_ms": tr,
                         "gpairs_per_s": pairs / t / 1e6, "tflops": flop / t / 1e9,
                         "fp32_peak_share": flop / t / 1e9 / info["fp32_fma_peak_tflops"]})
        tot, tot_ref = sum(r["ms"] for r in rows), sum(r["ref_ms"] for r in rows)
        res["forward"][f"B{B}"] = {"calls": rows, "ms_per_forward": tot, "ref_ms_per_forward": tot_ref}
        print(f"B={B}: {tot:.3f} ms per forward (28 graphs), reference ops {tot_ref:.3f} ms", flush=True)
    for C in (3, 64):
        x = torch.randn(16, N, C, generator=g).cuda()
        for k in (16, 17, 32, 33):
            out = torch.empty(16, N, k, dtype=torch.int64, device="cuda")
            kern = "register" if k <= 16 else "shared-memory list"
            res["boundary"][f"C{C}_k{k}"] = {"kernel": kern, "ms": timed(ours(x, k, out), a.warmup, a.reps)}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
