#!/usr/bin/env python
"""bench.py -- BA solver iterations/s on synthetic sliding windows (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--batch B] [--iters I] [--impl reference]
                    [--cams mono|stereo|quad] [--rho-sweep] [--swarm-agents A --swarms S] [--dump-outputs DIR]

A "step" = one solve of `iters` trust-region iterations (fixed schedule, convergence exits off so the
work per step is constant) on every window of the batch.  An iteration = one trust-region step attempt:
linearise all residuals (Jacobians + Huber), build and Schur-reduce the normal equations, solve the
reduced camera system, dogleg step, retract, evaluate the candidate, accept/reject -- the counting of
report.total_iterations (d2common/src/solver/SolverWrapper.cpp:41-42).

Workload at N=1 (BASELINE.json configs[1]): B independent single-drone 11-frame / 300-landmark windows
(W1, SURVEY.md 8d; 3000 reprojection + 10 IMU + 1 prior residual blocks each), distinct seeds.  The same line also
carries (a) `latency_b1`: one window through the reference-style reset -> add -> finalize -> solve -> read-back cycle,
(b) `swarm_1gpu`: the north-star case, 4-agent 11-frame / 300-landmark swarms with all agents as windows of one
handle on one GPU (ADMM, consensus reduced on the device) next to the CPU path with 4 threads and with all cores.
N>1 (configs[2], [3]): N-drone swarms, one agent per GPU, ADMM with the NCCL consensus exchange per sub-step; every rank
solves its agent's window of B swarms.  `--cams quad --rho-sweep` is config 4's quadcam / rho sweep mode.
`--dump-outputs DIR` writes what the last timed step handed back (see dump_outputs); the inputs are seeded, so two builds run
with the same arguments can be compared output for output.  Compare with a tolerance: the device's reductions are not
summed in a fixed order, and two runs of one build on a B200 (1000 W) differed by up to 1e-9 relative in the solved state.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from d2slam_b200 import abi, synth  # noqa: E402

OBS_BYTES = 176                      # SURVEY.md 8d: 20 f64 constants + 4 i32 ids
IMU_BYTES = 3736 + 3720
DUMP_LIMIT_BYTES = 64 << 20
DUMP_FILES = 8                       # pose, extrinsic, speed_bias, inv_depth, td, initial_cost, final_cost, window
RHO_SWEEP = [(1.0, 1.0), (10.0, 10.0), (100.0, 100.0), (1000.0, 1000.0), (10.0, 1000.0)]   # rho_T = rho_theta and one rho_T != rho_theta (consenus_factor.cpp:15-16)


def bytes_iter(pr):
    """Algorithmic bytes of one iteration of one window (SURVEY.md 8d BYTES_ITER)."""
    types = pr["obs"]["type"]
    p_of = {abi.PROJ_2F1C: (20, 2), abi.PROJ_2F2C: (26, 2), abi.PROJ_1F2C: (14, 2), abi.PROJ_2F1C_DEPTH: (20, 3), abi.PROJ_DEPTH_PRIOR: (1, 1)}
    b = 0
    for t, cnt in zip(*np.unique(types, return_counts=True)):
        p, d = p_of[int(t)]
        b += cnt * (OBS_BYTES + 8 * d * (p + 1))
    proj = b
    F = int(pr["n_own"]); npose = len(pr["frame_ids"]); C = len(pr["cam_ids"]); L = len(pr["lm_ids"])
    b += len(pr["imu"]) * IMU_BYTES
    if pr.get("prior") is not None:
        m = len(pr["prior"][1]); b += 8 * m * (m + 1)
    if pr.get("consensus") is not None:
        b += len(pr["consensus"][0]) * 8 * (13 + 6 * 7)
    n_c = 6 * npose + 9 * F
    b += 8 * (7 * (npose + C) + 9 * F + L + 1) + 8 * n_c * n_c
    return b, proj


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index = index; self.p = None; self.lines = []

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


@contextlib.contextmanager
def stdout_to_stderr():
    """NCCL announces its version on stdout when a communicator is created; the bench contract is ONE JSON line there."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        yield
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)


def host_threads_available():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def shared_per_pair(n_agents):
    """150 of an agent's 300 landmarks are co-observed by the other drones (SURVEY.md 8d W4), split evenly among them."""
    return max(1, 150 // max(1, n_agents - 1))


def make_batch(B, seed0, n_frames=11, n_landmarks=300, cams="mono"):
    return [synth.make_window(seed=seed0 + i, n_frames=n_frames, n_landmarks=n_landmarks, cams=cams) for i in range(B)]


def offset_slots(p, i, n_swarms):
    refs, slots, S = p["consensus"]
    q = synth.Problem(p)
    q["consensus"] = (refs, (slots + i * S).astype(np.int32), S * n_swarms)
    return q


def make_swarm_batch(B, seed0, n_agents, agents, cams="mono", distinct=None):
    """The windows of `agents` of B n_agents-drone swarms, swarm-major; swarm i uses the slot range [i*S, (i+1)*S).
    Only `distinct` different swarms are generated (the generator costs ~0.15 s per agent window); the rest are copies
    with their own buffers and slot ranges."""
    distinct = min(B, distinct or B)
    base = [synth.make_swarm(seed=seed0 + i, n_agents=n_agents, only_agents=list(agents), cams=cams, shared_per_pair=shared_per_pair(n_agents))
            for i in range(distinct)]
    out = []
    for i in range(B):
        for p in base[i % distinct]:
            out.append(offset_slots(p, i, B))
    return out


def load_all(solver, probs):
    for i, p in enumerate(probs):
        p.load(solver, i)


def reset_state(solver, probs):
    for i, p in enumerate(probs):
        solver.set_blocks(i, abi.POSE, p["frame_ids"], p["poses"], p["pose_const"])
        solver.set_blocks(i, abi.SPEED_BIAS, p["sb_ids"], p["sb"], None)
        solver.set_blocks(i, abi.LANDMARK, p["lm_ids"], p["inv_dep"], None)


def h2d_bytes(probs):
    b = 0
    for p in probs:
        b += p["obs"].nbytes + p["imu"].nbytes + p["poses"].nbytes + p["sb"].nbytes + p["inv_dep"].nbytes + p["ext"].nbytes
        if p.get("prior") is not None:
            b += p["prior"][0].nbytes + p["prior"][1].nbytes
    return int(b)


def d2h_bytes(probs):
    return int(sum(p["poses"].nbytes + p["sb"].nbytes + p["inv_dep"].nbytes for p in probs))


def dump_outputs(directory, get_blocks, probs, reps, suffix=""):
    """What the timed solve hands back to its caller, per window in batch order: the solved blocks (get_blocks(window, kind, ids))
    and the report's costs, concatenated over windows as float64 `<name><suffix>.npy`.  A batch whose outputs exceed 64 MB is
    reduced to a fixed, seeded sample of windows; `window.npy` lists the windows written."""
    per_window = [8 * (7 * (len(p["frame_ids"]) + len(p["cam_ids"])) + 9 * len(p["sb_ids"]) + len(p["lm_ids"]) + 4) for p in probs]
    budget = DUMP_LIMIT_BYTES - DUMP_FILES * 128      # an .npy header takes at most 128 bytes here (short names, 1-2 dims)
    keep = np.arange(len(probs))
    if sum(per_window) > budget:
        keep = np.sort(np.random.default_rng(0).permutation(len(probs))[: budget // max(per_window)])
    blocks = {"pose": (abi.POSE, "frame_ids"), "extrinsic": (abi.EXTRINSIC, "cam_ids"), "speed_bias": (abi.SPEED_BIAS, "sb_ids"), "inv_depth": (abi.LANDMARK, "lm_ids")}
    out = {name: np.concatenate([get_blocks(int(i), kind, probs[i][ids]) for i in keep]) for name, (kind, ids) in blocks.items()}
    out["inv_depth"] = out["inv_depth"][:, 0]
    out["td"] = np.array([get_blocks(int(i), abi.TD, np.zeros(1, np.int64))[0, 0] for i in keep])
    out["initial_cost"] = np.array([reps[i].initial_cost for i in keep])
    out["final_cost"] = np.array([reps[i].final_cost for i in keep])
    out["window"] = keep.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(directory, f"{name}{suffix}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def oracle_of(p, **cfg):
    from oracle import orc
    o = orc.Oracle(**cfg); p.load(o)
    return o


def cpu_sample(probs, iters, nthreads, max_windows):
    """Oracle (restated Ceres-equivalent CPU path, factors pinned to the reference's own classes) on a bounded sample."""
    from oracle import orc
    sample = probs[:max_windows]
    oras = [oracle_of(p, max_num_iterations=iters) for p in sample]
    t = time.perf_counter()
    reps = orc.solve_many(oras, nthreads, fixed_iters=iters)
    dt = time.perf_counter() - t
    its = sum(r.total_iterations for r in reps)
    return its / dt, len(sample), dt


def cpu_swarm_sample(swarms, iters, admm_steps, nthreads, max_swarms):
    """swarms: list of lists of Problem (one list per swarm). -> (iter/s, swarms used, seconds)"""
    from oracle import orc
    sample = swarms[:max_swarms]
    ags = [[oracle_of(p, max_num_iterations=iters, consensus_max_steps=admm_steps) for p in sw] for sw in sample]
    t = time.perf_counter()
    reps = orc.admm_many(ags, nthreads, fixed_mode=True)
    dt = time.perf_counter() - t
    return sum(r.total_iterations for r in reps) / dt, len(sample), dt


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank, world):
    """The reference's CPU implementation of the path on the host cores: the restated Ceres-equivalent solver whose
    factor arithmetic is pinned to the reference's own classes (oracle/_ref, tests/test_ref_pin.py); ceres::Solve itself is
    not available in this image.  One solver thread per window / swarm like ceres num_threads = 1, every host thread this
    process may run on busy, the GPU arm's window count per step (bounded when a step would take too long)."""
    if rank != 0:
        return
    from oracle import orc
    cores = host_threads_available()
    n_agents = max(1, args.gpus)
    iters = args.iters
    if n_agents == 1:
        n_units = args.batch
        probs = make_batch(n_units, 1000, cams=args.cams)
        oras = [oracle_of(p, max_num_iterations=iters) for p in probs]
        run = lambda m, nt=cores: orc.solve_many(oras[:m], nt, fixed_iters=iters)
        units = lambda m: list(zip(oras[:m], probs[:m]))
        workload = f"W1 single-drone 11-frame/300-landmark windows ({args.cams}), {iters} trust-region iterations per solve"
        unit = "windows"

        def restore(m):
            for o, p in zip(oras[:m], probs[:m]):
                o.set_blocks(abi.POSE, p["frame_ids"], p["poses"], p["pose_const"]); o.set_blocks(abi.SPEED_BIAS, p["sb_ids"], p["sb"], None)
                o.set_blocks(abi.LANDMARK, p["lm_ids"], p["inv_dep"], None)
    else:
        n_units = args.batch
        distinct = max(2, min(n_units, 2 * cores // n_agents, 32))
        base = [synth.make_swarm(seed=1000 + i, n_agents=n_agents, cams=args.cams, shared_per_pair=shared_per_pair(n_agents)) for i in range(distinct)]
        swarms = [[oracle_of(p, max_num_iterations=iters, consensus_max_steps=args.admm_steps) for p in base[i % distinct]] for i in range(min(n_units, 4 * distinct))]
        n_units = len(swarms)
        run = lambda m, nt=cores: orc.admm_many(swarms[:m], nt, fixed_mode=True)
        units = lambda m: [(o, p) for i, sw in enumerate(swarms[:m]) for o, p in zip(sw, base[i % distinct])]
        workload = (f"{n_agents}-drone swarm ({args.cams}), 11-frame/300-landmark windows + {(n_agents - 1) * 11} remote poses per agent, "
                    f"ADMM {args.admm_steps} sub-steps x {max(1, iters // args.admm_steps)} iterations")
        unit = "swarms"

        def restore(m):
            for sw, i in zip(swarms[:m], range(m)):
                for o, p in zip(sw, base[i % distinct]):
                    o.set_blocks(abi.POSE, p["frame_ids"], p["poses"], p["pose_const"]); o.set_blocks(abi.SPEED_BIAS, p["sb_ids"], p["sb"], None)
                    o.set_blocks(abi.LANDMARK, p["lm_ids"], p["inv_dep"], None)
    # parallel-efficiency self-check: a one-thread sample next to the all-thread run (a starved / cgroup-limited box shows here)
    m1 = max(1, min(n_units, 4 if n_agents == 1 else 1))
    t = time.perf_counter(); r1 = run(m1, 1); dt1 = time.perf_counter() - t
    one_thread = sum(r.total_iterations for r in r1) / dt1
    restore(m1)
    vals = []
    m_units, budget_s = n_units, 120.0   # the whole --steps / --warmup run has to end within a few minutes: bounded sample per step
    note = ""
    for s in range(args.warmup + args.steps):
        t = time.perf_counter()
        reps = run(m_units)
        dt = time.perf_counter() - t
        its = sum(r.total_iterations for r in reps)
        if s >= args.warmup:
            vals.append((its / dt, dt))
        if args.dump_outputs and s == args.warmup + args.steps - 1:
            u = units(m_units)
            dump_outputs(args.dump_outputs, lambda i, kind, ids: u[i][0].get_blocks(kind, ids), [p for _, p in u], reps)
        if s == 0 and dt * (args.warmup + args.steps) > budget_s:
            m_units = max(min(cores, n_units), int(n_units * budget_s / (dt * (args.warmup + args.steps))))
            note = f"; reduced to {m_units} {unit} per step after the first one to keep the run within {budget_s:.0f} s"
        restore(m_units)   # every step does the same work
    value = float(np.mean([v for v, _ in vals])); ms = float(np.mean([dt for _, dt in vals]) * 1e3)
    n_solves = m_units * (n_agents if n_agents > 1 else 1)
    sample = (f"{m_units} {unit} x {iters} iterations per step, one solver thread per {unit[:-1]} on {cores} host threads (sched_getaffinity){note}; "
              f"one thread alone: {one_thread:.0f} iter/s, parallel speed-up {value / one_thread:.1f}x")
    line = {
        "impl": "reference", "metric": "BA solver iterations/sec", "value": value, "unit": "iter/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload, "windows_per_gpu": args.batch, "solves_per_step": n_solves, "iters_per_solve": iters, "frames": 11, "landmarks": 300},
        "cpu_baseline": {"value": value, "unit": "iter/s", "cores": cores, "kind": "port", "one_thread_iter_s": one_thread, "parallel_speedup": value / one_thread,
                         "sample": sample + " (restated Ceres-equivalent DENSE_SCHUR+DOGLEG path, factor classes pinned to the reference's own sources; ceres itself cannot be built here)"},
        "e2e": {"value": value, "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ our arm: helpers
def timed_solves(solver, probs, iters, steps, warmup, barrier=None, step_barrier=None):
    """Device-resident throughput: problem already in HBM, only the (small) state is restored per step.
    -> (device seconds summed over steps [CUDA events on the solver stream], wall seconds, reports of the last step)"""
    for _ in range(warmup):
        reset_state(solver, probs); solver.solve_fixed(iters)
    if barrier:
        barrier()
    t0 = time.perf_counter()
    dev_ms = 0.0
    reps = None
    for _ in range(steps):
        reset_state(solver, probs)
        if step_barrier:
            step_barrier()   # ranks enter the solve together: the in-stream all-reduce otherwise waits out the peers' host-side jitter
        reps = solver.solve_fixed(iters)
        dev_ms += reps[0].total_time * 1e3
    if barrier:
        barrier()
    return dev_ms * 1e-3, time.perf_counter() - t0, reps


def latency_b1(local_rank, iters, cams):
    """One estimator, one window (the drop-in case): reset -> set_blocks/add_proj/add_imu/set_prior -> finalize -> solve -> get."""
    from d2slam_b200.harness import Replay
    from d2slam_b200.solver import Solver
    pr = synth.make_window(seed=4242, cams=cams)
    s1 = Solver(max_windows=1, device=local_rank, max_num_iterations=iters)
    rp = Replay([pr])
    rp.run(s1, 5, iters, 1)
    n = 30
    wall, reps = rp.run(s1, n, iters, 1)
    bd = {k: round(v / n * 1e3, 4) for k, v in rp.breakdown.items()}
    # a re-solve of the unchanged structure (graph replay): device time of the iterations alone
    dev = 1e9
    for _ in range(4):
        reset_state(s1, [pr])
        dev = min(dev, s1.solve_fixed(iters)[0].total_time * 1e3)
    s1.close()
    return {"ms": wall / n * 1e3, "device_ms_resolve": dev, "iters": iters, "iter_per_s": iters / (wall / n),
            "breakdown_ms": bd, "what": "B=1, W1 window, host buffers, reset -> add -> finalize -> solve -> read-back through the C ABI (C++ harness, one thread)"}


def consensus_gap(poses_by_agent, frame_ids_by_agent):
    """max distance between two agents' copies of the same frame position (the ADMM primal residual)."""
    seen = {}
    gap = 0.0
    for P, F in zip(poses_by_agent, frame_ids_by_agent):
        for p, f in zip(P, F):
            f = int(f)
            if f in seen:
                gap = max(gap, float(np.linalg.norm(p[:3] - seen[f])))
            else:
                seen[f] = p[:3]
    return gap


def swarm_one_gpu(args, local_rank, n_agents, n_swarms, iters, steps, warmup, cpu=True, rho=None, fixed=True):
    """All agents of n_swarms swarms as windows of ONE handle (consensus reduced on the device, no NCCL)."""
    from d2slam_b200.solver import Solver
    distinct = min(n_swarms, 37)
    probs = make_swarm_batch(n_swarms, 5000, n_agents, range(n_agents), cams=args.cams, distinct=distinct)
    cfg = dict(max_windows=len(probs), device=local_rank, max_num_iterations=iters, consensus_max_steps=args.admm_steps)
    if rho:
        cfg.update(rho_frame_T=rho[0], rho_frame_theta=rho[1])
    s = Solver(**cfg)
    load_all(s, probs); s.finalize()
    out = {"agents": n_agents, "swarms": n_swarms, "windows": len(probs), "obs_per_window": int(np.mean([len(p["obs"]) for p in probs[:n_agents]])),
           "pose_blocks_per_window": len(probs[0]["frame_ids"]), "admm_steps": args.admm_steps, "cams": args.cams}
    if not fixed:   # convergence exits on: iterations actually used + consensus gap (rho sweep)
        reset_state(s, probs)
        reps = s.solve()
        out["iterations_mean"] = float(np.mean([r.total_iterations for r in reps]))
        out["device_ms"] = reps[0].total_time * 1e3
        out["iter_per_s"] = float(sum(r.total_iterations for r in reps) / reps[0].total_time)
        out["consensus_gap_m"] = consensus_gap([s.get_blocks(i, abi.POSE, probs[i]["frame_ids"]) for i in range(n_agents)], [probs[i]["frame_ids"] for i in range(n_agents)])
        out["final_cost_mean"] = float(np.mean([r.final_cost for r in reps]))
        s.close()
        return out
    dev_s, wall_s, _ = timed_solves(s, probs, iters, steps, warmup)
    out["value"] = len(probs) * iters * steps / dev_s
    out["ms_per_step"] = dev_s / steps * 1e3
    reset_state(s, probs)
    out["kernel_ms_per_iteration"] = {k: round(v, 5) for k, v in s.kernel_times(iters).items()}
    # pose error against the oracle's in-process ADMM on swarm 0 (north star: <= 1e-4)
    from oracle import orc
    sw0 = probs[:n_agents]
    ags = [oracle_of(p, max_num_iterations=iters, consensus_max_steps=args.admm_steps, **({"rho_frame_T": rho[0], "rho_frame_theta": rho[1]} if rho else {})) for p in sw0]
    # the oracle's consensus table is per swarm: slots of swarm 0 are [0, S) already
    orc.admm_solve(ags, fixed_mode=True)
    reset_state(s, probs); s.solve_fixed(iters)
    dp = dr = 0.0
    for i, p in enumerate(sw0):
        a, b = synth.pose_errors(s.get_blocks(i, abi.POSE, p["frame_ids"]), ags[i].get_blocks(abi.POSE, p["frame_ids"]))
        dp, dr = max(dp, a), max(dr, b)
    out["pose_err_vs_oracle"] = {"pos_m": dp, "rot_rad": dr, "tolerance": 1e-4}
    # end to end from host buffers (sequential: feed -> finalize -> solve -> read back)
    from d2slam_b200.harness import Replay
    rp = Replay(probs)
    nth = max(1, min(host_threads_available(), 32))
    rp.run(s, 2, iters, nth)
    n = max(2, min(steps, 8))
    wall, _ = rp.run(s, n, iters, nth)
    out["e2e"] = {"value": len(probs) * iters * n / wall, "ms_per_step": wall / n * 1e3, "h2d_bytes_per_step": int(s.host_times()["h2d_bytes"]), "d2h_bytes_per_step": d2h_bytes(probs),
                  "breakdown_ms": {k: round(v / n * 1e3, 3) for k, v in rp.breakdown.items()}, "host_threads": nth, "handles_in_flight": 1}
    if cpu:
        swarms = [probs[i * n_agents:(i + 1) * n_agents] for i in range(n_swarms)]
        cores = host_threads_available()
        v4, n4, t4 = cpu_swarm_sample(swarms, iters, args.admm_steps, n_agents, min(len(swarms), 2 * n_agents))
        va, na, ta = cpu_swarm_sample(swarms, iters, args.admm_steps, cores, min(len(swarms), max(cores, n_agents)))   # every host thread gets a swarm
        out["cpu"] = {f"threads_{n_agents}": {"value": v4, "unit": "iter/s", "sample": f"{n4} swarms on {n_agents} host threads (one per agent: ceres num_threads = 1 per drone, d2vins_params.cpp:141,153; swarms solved concurrently so no thread idles at the consensus barrier), {t4:.1f} s"},
                      "all_cores": {"value": va, "unit": "iter/s", "cores": cores, "sample": f"{na} swarms on {cores} host threads, {ta:.1f} s"}}
        out["speedup"] = {f"device_vs_{n_agents}_threads": out["value"] / v4, "device_vs_all_cores": out["value"] / va,
                          f"e2e_vs_{n_agents}_threads": out["e2e"]["value"] / v4, "e2e_vs_all_cores": out["e2e"]["value"] / va}
    s.close()
    return out


# ------------------------------------------------------------------------------------------------ our arm
def pgo_leg(rank, world, local_rank, dist, cpu=True):
    """BASELINE configs[4] (SURVEY 8f rank 3): 10 000 poses on 8 trajectories, 40 000 relative-pose edges, Gauss-Newton with
    matrix-free block-Jacobi PCG; with N ranks the edges are sharded e % N and J^T J p is all-reduced over NCCL per CG iteration."""
    import torch
    from d2slam_b200 import pgo, synth
    g = pgo.make_pose_graph(seed=7, n_agents=8, poses_per_agent=1250, loops=30001)   # + 7 connecting closures = 40 000 edges
    sel = np.arange(rank, len(g["id_a"]), world)
    s = pgo.PgoSolver(device=local_rank, max_iterations=60, pcg_max_iterations=200, pcg_tolerance=1e-1, lambda0=1e-4, function_tolerance=1e-5)   # inexact LM: tools/pgo_sweep.py

    def load():
        s.set_poses(g["ids"], g["init"], g["fixed"]); s.add_edges(g["id_a"][sel], g["id_b"][sel], g["rel"][sel], g["sqrt_info"][sel])
    load()
    if world > 1:
        from d2slam_b200.solver import comm_unique_id
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.tensor(list(comm_unique_id()), dtype=torch.uint8))
        with stdout_to_stderr():
            dist.broadcast(uid, 0)
            s.comm_init(bytes(uid.cpu().tolist()), rank, world)
    s.solve()                     # warm-up (module load, first collectives)
    reps = []
    for _ in range(3):
        load()
        if dist is not None:
            torch.cuda.synchronize(); dist.barrier()
        reps.append(s.solve())
    r = min(reps, key=lambda q: q.device_ms)
    ms = torch.tensor([r.device_ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    x = s.get_poses(g["ids"])
    e0, _ = synth.pose_errors(g["init"], g["gt"]); e1, _ = synth.pose_errors(x, g["gt"])
    out = {"workload": f"{len(g['ids'])} poses / {len(g['id_a'])} edges (8 trajectories, odometry + loop closures), RelPoseFactorAD residual, Gauss-Newton + block-Jacobi PCG, edges sharded over {world} GPU(s)",
           "lm_iterations": r.iterations, "pcg_iterations": r.pcg_iterations, "device_ms": float(ms.item()), "ms_per_lm_iteration": float(ms.item()) / max(1, r.iterations),
           "lm_iterations_per_s": 1e3 * r.iterations / float(ms.item()), "initial_cost": r.initial_cost, "final_cost": r.final_cost, "converged": int(r.converged),
           "max_position_error_vs_ground_truth_m": {"initial_guess": e0, "solved": e1}}
    if cpu and rank == 0:
        from oracle import pgo_oracle as po
        t0 = time.perf_counter()
        _, costs = po.solve(g["init"], g["fixed"], g["ea"], g["eb"], g["rel"], g["sqrt_info"], iters=3)
        dt = time.perf_counter() - t0
        out["cpu_oracle"] = {"kind": "port", "what": "numpy linearisation + scipy sparse direct Gauss-Newton (oracle/pgo_oracle.py), 1 thread", "iterations": len(costs) - 1 if len(costs) > 1 else 1,
                             "s_per_iteration": dt / max(1, len(costs)), "cost_after": costs[-1]}
    s.close()
    return out


def run_ours(args, rank, world, local_rank):
    import torch
    from d2slam_b200.solver import Solver
    torch.cuda.set_device(local_rank)
    # feed threads + pinned staging on the GPU's NUMA node (what `numactl --cpunodebind` would do for the estimator process)
    from d2slam_b200 import hostaff
    bound_cpus = hostaff.bind_to_gpu_node(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        with stdout_to_stderr():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
    B, iters = args.batch, args.iters
    swarm = world > 1
    if swarm:
        # configs[2]/[3]: N-drone swarm, one agent per GPU, B swarms batched per GPU, ADMM consensus over NCCL
        probs = make_swarm_batch(B, 1000, world, [rank], cams=args.cams, distinct=74)
        solver = Solver(max_windows=B, device=local_rank, max_num_iterations=iters, consensus_max_steps=args.admm_steps)
    else:
        probs = make_batch(B, 1000 + rank * 100000, cams=args.cams)
        solver = Solver(max_windows=B, device=local_rank, max_num_iterations=iters)
    load_all(solver, probs)
    solver.finalize()
    if swarm:
        from d2slam_b200.solver import comm_unique_id
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.tensor(list(comm_unique_id()), dtype=torch.uint8))
        with stdout_to_stderr():
            dist.broadcast(uid, 0)
            solver.comm_init(bytes(uid.cpu().tolist()), rank, world)
            torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    parity = None
    if swarm:
        # correctness before timing: swarm 0 solved across the ranks (NCCL exchange) against the oracle's in-process ADMM
        reset_state(solver, probs); solver.solve_fixed(iters)
        mine = torch.from_numpy(solver.get_blocks(0, abi.POSE, probs[0]["frame_ids"])).cuda()
        allp = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allp, mine)
        if rank == 0:
            from oracle import orc
            sw0 = synth.make_swarm(seed=1000, n_agents=world, cams=args.cams, shared_per_pair=shared_per_pair(world))
            ags = [oracle_of(p, max_num_iterations=iters, consensus_max_steps=args.admm_steps) for p in sw0]
            orc.admm_solve(ags, fixed_mode=True)
            dp = dr = 0.0
            for a in range(world):
                x, y = synth.pose_errors(allp[a].cpu().numpy(), ags[a].get_blocks(abi.POSE, sw0[a]["frame_ids"]))
                dp, dr = max(dp, x), max(dr, y)
            parity = {"pos_m": dp, "rot_rad": dr, "tolerance": 1e-4, "what": f"swarm 0, {world} agents on {world} GPUs (NCCL consensus) vs the oracle's in-process ADMM, {iters} iterations"}
            if not (dp <= 1e-4 and dr <= 1e-4):
                sys.stderr.write(f"bench: multi-GPU parity check FAILED: {parity}\n")
        ok = torch.tensor([1 if (rank != 0 or (parity["pos_m"] <= 1e-4 and parity["rot_rad"] <= 1e-4)) else 0], device="cuda")
        dist.broadcast(ok, 0)
        if ok.item() != 1:
            dist.destroy_process_group()
            sys.exit(3)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t_dev, wall, last_reps = timed_solves(solver, probs, iters, args.steps, args.warmup, barrier, barrier if swarm else None)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, solver.get_blocks, probs, last_reps, f"_rank{rank}" if world > 1 else "")
    tt = torch.tensor([wall, t_dev], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    wall_max, dev_max = tt.tolist()
    total_iters = B * iters * args.steps * world
    value = total_iters / dev_max
    # ---- end to end through the C ABI with host buffers (C++ harness replaying D2Estimator's sequence):
    #      reset, add every block / residual, finalize (sort, tile, H2D), solve, read back the solved state (D2H)
    from d2slam_b200.harness import Replay
    rp = Replay(probs)
    ncpu = host_threads_available()
    # per pipeline stage: the feed and finalize stages of different handles run at the same time, so each gets a share of the cores
    seq_threads = max(1, min(ncpu // max(1, min(world, 8)), 32))           # one handle at a time: all the threads for its stage
    host_threads = seq_threads if (swarm or args.handles <= 2) else max(1, min(seq_threads, 12))
    if args.host_threads > 0:
        host_threads = args.host_threads
    e2e_steps = max(1, min(args.steps, 40))
    n_seq = min(e2e_steps, 10)
    rp.run(solver, 2, iters, seq_threads)
    barrier()
    seq_wall, _ = rp.run(solver, n_seq, iters, seq_threads)
    e2e_seq = {k: round(v / n_seq * 1e3, 3) for k, v in rp.breakdown.items()}
    e2e_seq["total_ms"] = round(seq_wall / n_seq * 1e3, 3)
    e2e_seq["iter_per_s"] = B * iters * n_seq / seq_wall
    if swarm:
        # the consensus handles own one NCCL communicator: keep the sequential driver here
        e2e_wall, e2e_breakdown, n_handles = seq_wall * e2e_steps / n_seq, dict(e2e_seq), 1
        barrier()
        h2d_step = solver.host_times()["h2d_bytes"]
    else:
        # consecutive steps overlapped across two independent handles: feed + finalize (k+1) | solve + read-back (k)
        n_handles = args.handles
        handles = [solver] + [Solver(max_windows=B, device=local_rank, max_num_iterations=iters) for _ in range(n_handles - 1)]
        rp.run_pipelined(handles, 2 * n_handles, iters, host_threads)
        barrier()
        e2e_wall, _ = rp.run_pipelined(handles, e2e_steps, iters, host_threads)
        e2e_breakdown = {"stage_busy_" + k.replace("_s", "_ms"): round(v / e2e_steps * 1e3, 3) for k, v in rp.breakdown.items()}
        e2e_breakdown["sequential_single_handle"] = e2e_seq
        e2e_breakdown["finalize_phases_ms"] = {k: v for k, v in solver.host_times().items() if k != "h2d_bytes"}
        barrier()
        h2d_step = solver.host_times()["h2d_bytes"]   # counted by the library: compact observation records + staging arena
        for hx in handles[1:]:
            hx.close()
    te = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = B * iters * e2e_steps * world / te.item()
    po, _, _ = rp.outputs(0, len(probs[0]["frame_ids"]), len(probs[0]["sb_ids"]), len(probs[0]["lm_ids"]))
    assert np.isfinite(po).all()
    # ---- per-kernel device times and roofline of the dominant kernel (CUDA events on the solver stream)
    reset_state(solver, probs)
    kt = solver.kernel_times(iters)
    rho_sweep = None
    if args.rho_sweep and swarm:
        # config 4: per rho the iterations actually used (convergence exits on), iter/s and the consensus gap after the solve
        rho_sweep = []
        for rT, rth in RHO_SWEEP:
            sx = Solver(max_windows=B, device=local_rank, max_num_iterations=iters, consensus_max_steps=args.admm_steps, rho_frame_T=rT, rho_frame_theta=rth)
            load_all(sx, probs); sx.finalize()
            if rank == 0:
                uid.copy_(torch.tensor(list(comm_unique_id()), dtype=torch.uint8))   # every handle owns its communicator
            with stdout_to_stderr():
                dist.broadcast(uid, 0)
                sx.comm_init(bytes(uid.cpu().tolist()), rank, world)
            sx.solve()          # warm-up: first collective on the new communicator, graph instantiation
            reset_state(sx, probs)
            barrier()
            reps = sx.solve()   # convergence exits on: the iterations each window actually used
            its = torch.tensor([float(sum(r.total_iterations for r in reps)), reps[0].total_time], dtype=torch.float64, device="cuda")
            mine = torch.from_numpy(sx.get_blocks(0, abi.POSE, probs[0]["frame_ids"])).cuda()
            allp = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allp, mine)
            fid = torch.from_numpy(np.asarray(probs[0]["frame_ids"], dtype=np.int64)).cuda()
            allf = [torch.zeros_like(fid) for _ in range(world)]
            dist.all_gather(allf, fid)
            tmax = its.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(its, op=dist.ReduceOp.SUM)
            cost = torch.tensor([float(np.mean([r.final_cost for r in reps]))], dtype=torch.float64, device="cuda")
            dist.all_reduce(cost, op=dist.ReduceOp.SUM)
            if rank == 0:
                rho_sweep.append({"rho_T": rT, "rho_theta": rth, "iter_per_s": its[0].item() / tmax[1].item(), "device_ms": tmax[1].item() * 1e3,
                                  "consensus_gap_m": consensus_gap([p.cpu().numpy() for p in allp], [f.cpu().numpy() for f in allf]),
                                  "final_cost_mean": cost.item() / world})
            sx.close()
    # pose-graph leg: collective (every rank holds a shard of the edges), so it runs before the non-zero ranks leave
    pg = pgo_leg(rank, world, local_rank, dist, cpu=False) if (world > 1 and not args.no_extras) else None
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    bi, proj_bytes = bytes_iter(probs[0])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s"
    dom = max(kt, key=kt.get)
    proj_gbs = B * proj_bytes / (kt["proj_lin"] * 1e-3) / 1e9
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = tj.get("proj_lin_pp_bytes_per_launch", tj.get("proj_lin_bytes_per_launch"))
        if traffic is not None:
            traffic = float(traffic) * B / float(tj.get("batch", B))   # captured at another batch size: scale per window
    except Exception:
        pass
    extra = {}
    if world == 1:
        # CPU baseline on rank 0, bounded sample, one thread (ceres_options.num_threads = 1)
        cpu_v, cpu_n, cpu_dt = cpu_sample(probs, iters, 1, min(B, args.cpu_windows))
        cpu_baseline = {"value": cpu_v, "unit": "iter/s", "cores": 1, "kind": "port",
                        "sample": f"{cpu_n} of the {B} windows x {iters} iterations, single thread ({cpu_dt:.1f} s); factor classes of the port pinned to the reference's own sources (oracle/_ref)"}
        solver.close()
        if not args.no_extras:
            extra["latency_b1"] = latency_b1(local_rank, iters, args.cams)
            sw = swarm_one_gpu(args, local_rank, args.swarm_agents, args.swarms, iters, max(3, min(args.steps, 10)), 3)
            extra["swarm_1gpu"] = sw
            if args.rho_sweep:
                extra["rho_sweep_1gpu"] = [dict(rho_T=r[0], rho_theta=r[1], **swarm_one_gpu(args, local_rank, args.swarm_agents, max(1, args.swarms // 4), iters, 3, 1, cpu=False, rho=r, fixed=False))
                                           for r in RHO_SWEEP]
    else:
        cpu_baseline = {"value": None, "unit": "iter/s", "cores": 0, "kind": "port", "sample": "timed at N=1 only (bench contract)"}
    if not args.no_extras:
        extra["pgo"] = pg if world > 1 else pgo_leg(rank, world, local_rank, dist, cpu=True)
    n_variants = len(set(int(t) for t in np.unique(probs[0]["obs"]["type"]))) if args.cams != "mono" else 1
    # per solve: tr_reset, misc_lin, proj_lin, control (+ per ADMM sub-step: memset, cons_pack, cons_apply, cons_refs, tr_reset);
    # per iteration: lm_gather, sb_elim, schur (1-2 launches), leaf_elim, chol, sb_back, leaf_back, step, misc_lin, proj_lin (n_variants), control
    per_iter = (8 + n_variants) if not swarm else (11 + n_variants)
    launches = args.steps * (3 + n_variants + (args.admm_steps * (5 + 2 + n_variants) if swarm else 0) + iters * per_iter)
    line = {
        "metric": "BA solver iterations/sec", "value": value, "unit": "iter/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_max * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": (f"{world}-drone swarm ({args.cams}), 11-frame/300-landmark windows + {(world - 1) * 11} remote poses per agent ({shared_per_pair(world)} landmarks shared per drone pair), one agent per GPU, "
                                f"{B} swarms batched, ADMM {args.admm_steps} sub-steps x {max(1, iters // args.admm_steps)} iterations, NCCL all-reduce consensus" if swarm else
                                f"W1 single-drone 11-frame/300-landmark windows ({args.cams}; configs[1]); batch of {B} independent windows per GPU, "
                                f"{iters} trust-region iterations per solve, fixed schedule"),
                   "windows_per_gpu": B, "iters_per_solve": iters, "frames": 11, "landmarks": 300, "residual_blocks": len(probs[0]["obs"]) + 11,
                   "l2_policy": "inputs larger than L2 (batch working set >> 126 MB)" if B >= 128 else "batch smaller than L2",
                   "wall_ms_per_step": wall_max * 1e3 / args.steps, "bytes_iter_per_window": int(bi),
                   "weak_scaling_note": ("the per-GPU work GROWS with N: an agent's window holds 11 own + 11 (N-1) remote pose blocks and the cross-drone observations, so "
                                         "value(N) / (N value(1)) mixes hardware scaling with a larger problem per GPU") if swarm else None},
        "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": "iter/s", "h2d_bytes_per_step": int(h2d_step), "host_input_bytes_per_step": h2d_bytes(probs), "d2h_bytes_per_step": d2h_bytes(probs),
                "steps": e2e_steps, "host_threads": host_threads, "host_threads_sequential_leg": seq_threads, "handles_in_flight": n_handles, "numa_bound_cpus": bound_cpus,
                "ms_per_step_breakdown": e2e_breakdown,
                "note": "every step runs the full C-ABI sequence from HOST buffers: d2ba_reset + set_blocks/add_proj/add_imu/set_prior_info + d2ba_finalize (order, tile plan, pinned H2D) + d2ba_solve_fixed + d2ba_get_blocks (D2H), driven by the C++ harness; with handles_in_flight > 1 consecutive steps overlap on independent handles"},
        "roofline": {"bound": "hbm", "kernel": "k_proj_lin_pp (reprojection linearisation + group J^T J)", "achieved": proj_gbs, "peak": peak, "unit": "GB/s", "frac": proj_gbs / peak,
                     "traffic": traffic, "peak_source": peak_src, "dominant_kernel_by_time": dom,
                     "algorithmic_bytes_per_launch": int(B * proj_bytes), "kernel_ms_per_iteration": kt,
                     "whole_iteration_frac": B * bi / (sum(kt.values()) * 1e-3) / 1e9 / peak},
        "cpu_baseline": cpu_baseline,
        "clocks": clocks,
    }
    if parity is not None:
        line["parity_check"] = parity
    if rho_sweep is not None:
        line["rho_sweep"] = rho_sweep
    line.update(extra)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=592)   # 4 x 148 SMs: whole waves of the one-CTA-per-window kernels
    ap.add_argument("--iters", type=int, default=8)
    ap.add_argument("--cpu-windows", type=int, default=96)
    ap.add_argument("--admm-steps", type=int, default=4)
    ap.add_argument("--cams", default="mono", choices=["mono", "stereo", "quad"])
    ap.add_argument("--rho-sweep", action="store_true")
    ap.add_argument("--swarm-agents", type=int, default=4)   # north-star leg at N=1: 4-agent swarms on one GPU
    ap.add_argument("--swarms", type=int, default=148)
    ap.add_argument("--handles", type=int, default=4)
    ap.add_argument("--host-threads", type=int, default=0, help="feeding / planning threads per stage of the e2e leg (0 = min(cores, 32))")
    ap.add_argument("--no-extras", action="store_true", help="N=1: skip the latency_b1 / swarm_1gpu legs")
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's solved state and costs as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # watchdog: a rank stuck in a collective must not hang the launcher -- dump every thread's Python stack and exit
    import faulthandler
    faulthandler.enable()
    wd = int(os.environ.get("D2BA_BENCH_WATCHDOG", "0")) or (600 if world > 1 else 0)
    if wd > 0:
        faulthandler.dump_traceback_later(wd, exit=True)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
