"""bench.py's reference arm (the CPU port timed on the host cores): the JSON line carries every key the
bench contract names, and under a multi-rank launch only rank 0 prints.  No GPU involved, except in
test_dump_outputs_writes_every_pair_record (the GPU arm on a short sequence)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env):
    env = dict(os.environ, MV_BENCH_REF_BUDGET_S="0.3", **extra_env)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus",
                        extra_env.get("WORLD_SIZE", "1"), "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_line_has_the_contract_keys():
    lines = _run({})
    assert len(lines) == 1
    d = lines[0]
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["data"] == "synthetic"
    assert d["metric"].startswith("frame-pairs/sec") and d["unit"] == "frame-pairs/s"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_print_nothing():
    assert _run({"WORLD_SIZE": "2", "RANK": "1", "LOCAL_RANK": "1"}) == []


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 2 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_writes_every_pair_record(tmp_path):
    n_frames = 9
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                        "--frames", str(n_frames), "--no-e2e", "--no-cpu", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")][0]
    assert line["steps"] == 2
    shapes = {"q": (8, 4), "t": (8, 3), "pnp_inliers": (8,), "pnp_cost": (8,), "num_matches": (8,),
              "ransac_inliers": (8,), "best_hypothesis": (8,), "status": (8,)}
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(k + ".npy" for k in shapes)
    for name, shape in shapes.items():
        a = np.load(tmp_path / (name + ".npy"))
        assert a.shape == shape and a.dtype in (np.float32, np.float64), name
    n = np.load(tmp_path / "num_matches.npy")
    assert (n == np.round(n)).all() and n.sum() > 0
    assert line["run"]["mean_matches_per_pair"] == n.sum() / (n_frames - 1)
    # the dumped records against the CPU oracle on the same seeded frames (its own generator): counts and the
    # selected hypothesis exactly, the pose within the benchmark's tolerance
    import bench
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import synth
    from oracle import orc
    o = orc.Oracle()
    offs = synth.default_offsets(n_frames, bench.SEED)
    frames = [o.synth_frame(bench.SEED, bench.ROWS, bench.COLS, f, int(offs[f, 0]), int(offs[f, 1]))
              for f in range(n_frames)]
    cfg = bench.track_cfg_for_oracle(orc, synth)
    ref = [o.track_pair(cfg, p, *frames[p], *frames[p + 1][:2]) for p in range(n_frames - 1)]
    dumped = {k: np.load(tmp_path / (k + ".npy")) for k in shapes}
    got = [{k: v[p] for k, v in dumped.items()} for p in range(n_frames - 1)]
    parity = bench.parity_against_port(got, ref, n_frames - 1)
    assert parity["mismatches"] == 0, parity
