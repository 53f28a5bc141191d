"""L1 on the device against the REFERENCE's own factor classes (oracle/_ref/libd2ref.so: the unmodified D2SLAM sources
compiled by oracle/Makefile.ref): every reprojection / IMU / consensus factor of seeded windows -- the CUDA path's residual
and tangent Jacobian vs ProjectionTwoFrame*Factor::Evaluate, IMUFactor::Evaluate, ConsenusPoseFactor::Evaluate.

Where the library is absent the reprojection and IMU answers come from tests/golden/ref_extra.npz (the same library on the
same seeded windows, tests/golden/make_ref_golden.py; a fixed sample of the reprojection factors), and the consensus factor is
the oracle's, which tests/test_ref_pin.py pins to ConsenusPoseFactor at 1e-14 on frozen reference vectors."""
import os

import numpy as np
import pytest

from d2slam_b200 import abi, synth
from oracle import ref

pytestmark = pytest.mark.gpu
HAVE_REF = ref.available()
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_extra.npz")

PROJ_CASES = [dict(seed=2, cams="stereo", estimate_extrinsic=True, estimate_td=True, td_offset=0.002, n_landmarks=60, n_frames=5),
              dict(seed=5, cams="quad", n_landmarks=80, n_frames=4)]
IMU_CASE = dict(seed=9, n_landmarks=40, n_frames=6)
# device layout of a reprojection record's Jacobian: [pose_i 6 | pose_j 6 | ext_a 6 | ext_b 6 | lambda | td]
PROJ_BLOCKS = {abi.PROJ_2F1C: [(0, 0), (6, 1), (12, 2)], abi.PROJ_2F2C: [(0, 0), (6, 1), (12, 2), (18, 3)], abi.PROJ_1F2C: [(12, 0), (18, 1)]}


def scaled(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(b).max(), 1.0))


def proj_sample(pr, per_type=24):
    """The reprojection factors frozen for machines without the library: up to `per_type` of every factor type."""
    rng = np.random.default_rng(0)
    types = pr["obs"]["type"]
    return np.sort(np.concatenate([rng.permutation(np.flatnonzero(types == t))[:per_type] for t in np.unique(types)]))


def reference_proj(pr, idx):
    """The reference classes on observations `idx` of window `pr` -> residuals [n, 2], Jacobians [n, 2, 26] in the device layout."""
    pose = {int(i): p for i, p in zip(pr["frame_ids"], pr["poses"])}
    ext = {int(i): p for i, p in zip(pr["cam_ids"], pr["ext"])}
    lam = {int(i): v for i, v in zip(pr["lm_ids"], pr["inv_dep"])}
    td = np.array([pr["td"]])
    R = np.zeros((len(idx), 2)); J = np.zeros((len(idx), 2, 26))
    for n, k in enumerate(idx):
        o = pr["obs"][k]
        t = int(o["type"])
        pi, pj, ea, eb = pose[int(o["frame_a"])], pose.get(int(o["frame_b"])), ext[int(o["cam_a"])], ext.get(int(o["cam_b"]))
        l = np.array([lam[int(o["landmark_id"])]])
        params = {abi.PROJ_2F1C: [pi, pj, ea, l, td], abi.PROJ_2F2C: [pi, pj, ea, eb, l, td], abi.PROJ_1F2C: [ea, eb, l, td]}[t]
        r, Js, _ = ref.proj_eval(t, o["pts_i"], o["pts_j"], o["vel_i"], o["vel_j"], float(o["td_i"]), float(o["td_j"]), 0.0, params)
        R[n] = r
        for off, bi in PROJ_BLOCKS[t]:
            assert np.all(Js[bi][:, 6] == 0)
            J[n, :, off:off + 6] = Js[bi][:, :6]
        J[n, :, 24] = Js[-2][:, 0]; J[n, :, 25] = Js[-1][:, 0]
    return R, J


def reference_imu(pr):
    """The reference IMUFactor on every IMU factor of `pr` -> residuals [n, 15], Jacobians [n, 15, 30] (tangent), sqrt_info [n, 15, 15]."""
    pose = {int(i): p for i, p in zip(pr["frame_ids"], pr["poses"])}
    sb = {int(i): p for i, p in zip(pr["sb_ids"], pr["sb"])}
    R, J, SI = [], [], []
    for m in pr["imu"]:
        pre = {f: m[f] for f in ("sum_dt", "delta_p", "delta_q", "delta_v", "jacobian", "covariance")}
        r, Js, si = ref.imu_eval(pre, m["linearized_ba"], m["linearized_bg"], pose[int(m["frame_a"])], sb[int(m["frame_a"])], pose[int(m["frame_b"])], sb[int(m["frame_b"])])
        R.append(r); J.append(np.concatenate([Js[0][:, :6], Js[1], Js[2][:, :6], Js[3]], axis=1)); SI.append(si)
    return np.array(R), np.array(J), np.array(SI)


@pytest.mark.parametrize("case", PROJ_CASES)
def test_reprojection_factors_on_device_match_reference_classes(case):
    from d2slam_b200.solver import Solver
    pr = synth.make_window(**case)
    s = Solver(); pr.load(s, 0); s.finalize(); s.debug_linearize()
    dev = s.debug_get(0, abi.DBG_PROJ_RESJAC).reshape(-1, 81)
    if HAVE_REF:
        idx = np.arange(len(pr["obs"]))
        r_ref, J_ref = reference_proj(pr, idx)
    else:
        c = PROJ_CASES.index(case)
        g = np.load(GOLD)
        idx = proj_sample(pr)
        assert np.array_equal(idx, g[f"dev_proj{c}_idx"])
        r_ref, J_ref = g[f"dev_proj{c}_r"], g[f"dev_proj{c}_J"]
    worst = 0.0
    seen = set()
    for n, k in enumerate(idx):
        t = int(pr["obs"][k]["type"]); seen.add(t)
        d = dev[k]; J = d[3:].reshape(3, 26)[:2]
        worst = max(worst, scaled(d[:2], r_ref[n]))
        for off, _ in PROJ_BLOCKS[t]:
            worst = max(worst, scaled(J[:, off:off + 6], J_ref[n][:, off:off + 6]))
        worst = max(worst, scaled(J[:, 24], J_ref[n][:, 24]), scaled(J[:, 25], J_ref[n][:, 25]))
    assert worst <= 1e-12, worst
    assert len(seen) >= 2


def test_imu_factors_on_device_match_reference_class():
    from d2slam_b200.solver import Solver
    pr = synth.make_window(**IMU_CASE)
    s = Solver(); pr.load(s, 0); s.finalize(); s.debug_linearize()
    dev = s.debug_get(0, abi.DBG_IMU_RESJAC).reshape(-1, 465)
    assert len(dev) == len(pr["imu"]) > 0
    if HAVE_REF:
        r_ref, J_ref, si_ref = reference_imu(pr)
    else:
        g = np.load(GOLD)
        r_ref, J_ref, si_ref = g["dev_imu_r"], g["dev_imu_J"], g["dev_imu_sqrt_info"]
    for k in range(len(pr["imu"])):
        J = dev[k][15:].reshape(15, 30)
        # sqrt_info = LLT(cov^-1)^T of a 1e8-conditioned covariance: compare un-whitened (1e-10) and whitened (1e-7)
        U = np.linalg.inv(si_ref[k])
        assert scaled(U @ dev[k][:15], U @ r_ref[k]) <= 1e-10 and scaled(U @ J, U @ J_ref[k]) <= 1e-10
        assert scaled(dev[k][:15], r_ref[k]) <= 1e-7 and scaled(J, J_ref[k]) <= 1e-7


def test_consensus_factors_on_device_match_reference_class():
    from d2slam_b200.solver import Solver
    from test_ref_pin import orc_cons
    sw = synth.make_swarm(seed=12, n_agents=3, n_landmarks=60, shared_per_pair=20, n_frames=5)
    cfg = dict(consensus_max_steps=2, max_num_iterations=4, rho_frame_T=10.0, rho_frame_theta=1000.0)
    s = Solver(max_windows=3, **cfg)
    for i, p in enumerate(sw):
        p.load(s, i)
    s.finalize(); s.solve_fixed(4)       # leaves z, tilde of the last sub-step and the solved x on the device
    n = 0
    for i in range(3):
        rec = s.debug_get(i, abi.DBG_CONS_RESJAC).reshape(-1, 62)
        for q in rec:
            if not np.any(q):
                continue
            x, z, tl, r, J = q[:7], q[7:14], q[14:20], q[20:26], q[26:].reshape(6, 6)
            if HAVE_REF:
                rr, Jr = ref.consensus_eval(z[:3], z[3:7], tl[:3], tl[3:], cfg["rho_frame_T"], cfg["rho_frame_theta"], x)
            else:
                rr, Jr = orc_cons(dict(z=z.copy(), x=x.copy(), tt=tl[:3].copy(), th=tl[3:].copy(), rho_T=cfg["rho_frame_T"], rho_theta=cfg["rho_frame_theta"]))
            assert scaled(r, rr) <= 1e-13 and scaled(J, Jr[:, :6]) <= 1e-13
            n += 1
    assert n >= 30
