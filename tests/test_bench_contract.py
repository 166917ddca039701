"""bench.py contract pieces: the reference arm's JSON line and the helpers (CPU), --dump-outputs (CPU and GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--ref-batch", "4"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_algorithmic_bytes_and_measured_traffic_helpers():
    sys.path.insert(0, ROOT)
    import bench
    alg = bench.algorithmic(96, 256, 0, 4, 10.0)
    # north_star: (K+1) x (m^2 + mn + n^2) x 4 B per solve
    assert alg["b_fwd_stream"] == 11 * (256 * 256 + 256 * 96 + 96 * 96) * 4
    assert alg["W_fwd"] > 1e8 and alg["b_fwd_resident"] < alg["b_fwd_stream"]
    t = bench.measured_traffic(4096)
    assert t is None or t > 1e9            # bytes per forward launch from the newest profiles/*_fwd_traffic.json
    assert bench.measured_traffic(2048) is None or abs(bench.measured_traffic(2048) * 2 - t) < 1.0


def test_world_reference_arm_and_scene_generators():
    """--config world reference arm (oracle world on the host) prints the contract line; the config-4 / world initial
    conditions are piles in contact from step 0 (what the bench lines claim)."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "world",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["unit"] == "world-steps/s" and d["value"] > 0 and d["gpu_launches"] == 0
    sys.path.insert(0, ROOT)
    import bench
    from oracle.world_oracle import OracleCircleWorld
    ic = bench.world_initial(2, 0)
    assert ic["pos"].shape == (2, 25, 2)
    w = OracleCircleWorld(ic["pos"][1], ic["rad"][1], ic["vel"][1], ic["mass"][1], ic["rest"][1], ic["fric"][1],
                          gravity=100.0, static=(0,), dt=1.0 / 30)
    assert 40 <= len(w.contacts) <= 75                       # 24-ball pile: ~51 contacts, within BatchedWorld's default capacity
    ic4 = bench.cfg4_initial(1, 0)
    assert ic4["pos"].shape == (1, 513, 2) and float(ic4["rad"][0, 1]) == 10.0
    # neighbours of the hexagonal pile are closer than eps = 0.1: in contact before the first step
    d01 = (ic4["pos"][0, 1] - ic4["pos"][0, 2]).norm() - 20.0
    assert 0.0 < float(d01) < 0.1


def test_dump_outputs_keeps_one_seeded_sample_of_scenes_under_64_mb(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    B = 4096
    big = torch.randn(B, 64, 64, dtype=torch.float64)          # 32 KB per scene, 134 MB in all
    scene = torch.arange(B, dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / "a"), {"big": big, "scene": scene, "absent": None})
    bench.dump_outputs(str(tmp_path / "b"), {"big": big, "scene": scene})
    assert sorted(os.listdir(tmp_path / "a")) == ["big.npy", "scene.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 * 10 ** 6
    kept = np.load(tmp_path / "a" / "scene.npy")
    assert kept.dtype == np.float64 and 0 < len(kept) < B and (np.diff(kept) > 0).all()
    assert np.array_equal(np.load(tmp_path / "a" / "big.npy"), big[torch.from_numpy(kept).long()].numpy())
    assert np.array_equal(np.load(tmp_path / "b" / "scene.npy"), kept)


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """--dump-outputs writes every result of the timed path; at 64 scenes all of them, in the run's dtype."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", "64", "--steps", "2", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["steps"] == 2 and d["gpu_launches"] == 8
    shapes = {"zhat": (64, 96), "lam": (64, 256), "slack": (64, 256), "status": (64,), "iters": (64,), "resid": (64,),
              "grad_Q": (64, 96, 96), "grad_p": (64, 96), "grad_G": (64, 256, 96), "grad_h": (64, 256),
              "grad_F": (64, 256, 256)}
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in shapes)
    z = {k: np.load(tmp_path / (k + ".npy")) for k in shapes}
    for k, s in shapes.items():
        assert z[k].shape == s and z[k].dtype == (np.float64 if k in ("status", "iters") else np.float32), k
    sys.path.insert(0, ROOT)
    from lcp_physics_b200 import solve_forward
    from lcp_physics_b200.scenes import make_scenes
    inp = make_scenes(64, 32, 64, fd=2, e=0, dtype=torch.float32, seed=1000)
    zhat = solve_forward(*(t.cuda() for t in inp), max_iter=10)[0].cpu().double()
    err = (torch.from_numpy(z["zhat"]).double() - zhat).norm(dim=1) / zhat.norm(dim=1)
    assert float(err.max()) < 1e-5
