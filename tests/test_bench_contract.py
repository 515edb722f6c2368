"""bench.py's reference arm runs on the CPU: check here that it prints exactly ONE JSON line on stdout with the keys the
driver reads (the B200 arm shares the emit path; its numbers are checked on the GPU box)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=REPO)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "pgd_attack_steps_per_sec" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    cb = d["cpu_baseline"]
    from oracle import build_ref
    assert cb["kind"] == ("reference" if build_ref.available() else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "B=16x4096" in d["config"]["workload"]
    import bench
    assert d["config"] == bench.config_dict()          # both arms print the same config
    adv = np.load(tmp_path / "adv.npy")
    x, _, _ = bench.make_inputs(bench.B_PER_GPU, 0)
    assert adv.dtype == np.float32 and adv.shape == tuple(x.shape)
    assert np.array_equal(adv[:, :3], x[:, :3].numpy()) and not np.array_equal(adv[:, 3:6], x[:, 3:6].numpy())


@pytest.mark.gpu
def test_native_arm_dumps_what_the_timed_attack_returned(tmp_path):
    """--steps K times tar_NB_attack(iters=K), and --dump-outputs writes that attack's result: the same call made here on
    the same seeded inputs gives the same array."""
    import torch
    K = 3
    p = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", str(K), "--warmup", "0", "--repeats", "1",
                        "--mlp", "tf32", "--no-cpu", "--no-parity", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=REPO)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout)
    assert d["steps"] == K and d["timing"]["steps_per_repeat"] == K
    import bench
    from pointsecguard_b200 import synthetic as syn, torchattacks
    from pointsecguard_b200.engine import MLP_TF32
    from pointsecguard_b200.models.pointnet2_sem_seg import get_model
    model = get_model(13)
    model.load_state_dict(syn.make_state_dict("ssg", init="he"))
    model = model.cuda().eval()
    model.set_mlp_mode(MLP_TF32)
    x, labels, mask = bench.make_inputs(bench.B_PER_GPU, 0)
    torch.manual_seed(0)
    want = torchattacks.tar_NB_attack(model, eps=bench.EPS, alpha=bench.ALPHA, iters=K, target=bench.TARGET, mask=mask)(
        x.cuda(), labels.numpy().astype(np.float64))
    got = np.load(tmp_path / "adv.npy")
    assert got.dtype == np.float32 and np.array_equal(got, want.cpu().numpy())


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=REPO, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""
