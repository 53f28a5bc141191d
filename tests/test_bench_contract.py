"""bench.py contract (the reference arm runs on CPU: no GPU needed; the device path's --dump-outputs test needs one)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--batch", "8"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "BA solver iterations/sec" and d["unit"] == "iter/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == "iter/s" and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_collective_legs_run_before_the_non_zero_ranks_leave():
    """The pose-graph leg all-reduces across every rank: it must sit before the early return of rank != 0 in run_ours
    (a rank-0-only call hangs the launcher -- found the hard way at N = 2)."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    body = src[src.index("def run_ours("):src.index("def main(")]
    leave = body.index("if rank != 0:")
    multi = body.index("pgo_leg(rank, world, local_rank, dist, cpu=False)")
    assert multi < leave
    # after the return only rank 0 is left: nothing collective may follow for world > 1
    tail = body[leave:]
    assert "pg if world > 1 else pgo_leg" in tail and "dist.all_reduce" not in tail and "dist.barrier" not in tail and "dist.broadcast" not in tail


def test_dump_outputs_writes_the_solved_state_and_repeats_run_to_run(tmp_path):
    """--dump-outputs: the last timed step's solved blocks and costs as float64 .npy; seeded inputs, so two runs agree."""
    import numpy as np
    dumps = []
    for k in range(2):
        d = tmp_path / str(k)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0", "--batch", "2",
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        dumps.append({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = dumps
    assert set(a) == {"pose", "extrinsic", "speed_bias", "inv_depth", "td", "initial_cost", "final_cost", "window"}
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["pose"].shape == (22, 7) and a["speed_bias"].shape == (22, 9) and a["inv_depth"].shape == (600,) and np.array_equal(a["window"], [0, 1])
    assert np.all(a["final_cost"] < a["initial_cost"])
    for k in a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.gpu
def test_dump_outputs_of_the_device_path_hold_the_solved_windows(tmp_path):
    """--dump-outputs on the timed CUDA path: the last step's solved state of every window, equal to the oracle's solve of the
    same seeded windows (bench.make_batch) with the same fixed schedule."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from d2slam_b200 import abi, synth
    from oracle import orc
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", "2", "--steps", "2", "--warmup", "1", "--iters", "6", "--no-extras",
                          "--cpu-windows", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = {f[:-4]: np.load(tmp_path / f) for f in sorted(os.listdir(tmp_path))}
    assert set(d) == {"pose", "extrinsic", "speed_bias", "inv_depth", "td", "initial_cost", "final_cost", "window"}
    assert all(v.dtype == np.float64 for v in d.values()) and np.array_equal(d["window"], [0, 1])
    probs = bench.make_batch(2, 1000)
    assert d["pose"].shape == (22, 7) and d["speed_bias"].shape == (22, 9) and d["inv_depth"].shape == (600,)
    for i, p in enumerate(probs):
        o = orc.Oracle(max_num_iterations=6); p.load(o)
        rep = o.solve_fixed(6)
        dp, dr = synth.pose_errors(d["pose"][11 * i:11 * (i + 1)], o.get_blocks(abi.POSE, p["frame_ids"]))
        assert dp < 1e-6 and dr < 1e-6, (i, dp, dr)
        assert abs(d["final_cost"][i] - rep.final_cost) <= 1e-6 * max(1.0, rep.final_cost)
        assert abs(d["initial_cost"][i] - rep.initial_cost) <= 1e-8 * max(1.0, rep.initial_cost)
        assert np.abs(d["inv_depth"][300 * i:300 * (i + 1)] / o.get_blocks(abi.LANDMARK, p["lm_ids"])[:, 0] - 1).max() < 1e-6
