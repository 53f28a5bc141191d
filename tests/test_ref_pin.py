"""Pins the oracle's restated factors (oracle/orc_factors.c) to the REFERENCE's own classes.

oracle/_ref/libd2ref.so holds the unmodified reference sources (d2vins/src/factors/projection*Factor.cpp, imu_factor.h +
d2common integration_base.h / utils.hpp, d2common/src/solver/consenus_factor.cpp, pose_local_parameterization.cpp)
compiled by oracle/Makefile.ref against the stand-in third-party headers of oracle/_shim.  Every comparison is
reference Evaluate() vs orc_*_eval on the same seeded inputs: residuals and every Jacobian block, <= 1e-12 of the block's
scale (both sides are f64 with different but equivalent operation orders; sqrt_info = 307 amplifies rounding).
The same reference outputs are frozen in tests/golden/ref_factors.npz and tests/golden/ref_extra.npz
(tests/golden/make_ref_golden.py): where the library is absent every test compares with those instead.
"""
import ctypes as C
import os

import numpy as np
import pytest

from d2slam_b200 import abi, synth
from oracle import orc, ref

import test_oracle_factors as tof

L = orc.lib()
HAVE_REF = ref.available()
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_factors.npz")
GOLD_EXTRA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_extra.npz")


def frozen():
    """The library's answers on the seeded cases below (tests/golden/make_ref_golden.py)."""
    g, x = np.load(GOLD), np.load(GOLD_EXTRA)
    return {**{k: g[k] for k in g.files}, **{k: x[k] for k in x.files}}


def close(a, b, tol=1e-12):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(np.abs(b).max(), 1.0)
    err = np.abs(a - b).max() / scale
    assert err <= tol, err
    return err


# ----------------------------------------------------------------------------------------------- case generators (seeded)
def proj_cases(seed=7, n=6):
    rng = np.random.default_rng(seed)
    tof.RNG = np.random.default_rng(seed + 1)
    out = []
    for typ in (abi.PROJ_2F1C, abi.PROJ_2F2C, abi.PROJ_1F2C, abi.PROJ_2F1C_DEPTH):
        for k in range(n):
            pi, pj, ea, eb, Pw, bi, lam = tof.scene()
            ext_j = eb if typ in (abi.PROJ_2F2C, abi.PROJ_1F2C) else ea
            pose_j = pi if typ == abi.PROJ_1F2C else pj
            bj, dj = synth._bearing(Pw[None], pose_j, ext_j)
            bj = bj[0] + rng.normal(size=3) * 2e-3; bj /= np.linalg.norm(bj)
            vel_i = rng.normal(size=3) * 0.05; vel_j = rng.normal(size=3) * 0.05
            td_i, td_j = (0.0, 0.0) if k % 2 == 0 else (0.001, -0.002)
            td = 0.0 if k % 3 == 0 else 0.003
            out.append(dict(typ=typ, pi=pi, pj=pj, ea=ea, eb=eb, lam=lam * (1.0 + 0.1 * rng.normal()), td=td, pts_i=bi, pts_j=bj, vel_i=vel_i, vel_j=vel_j,
                            td_i=td_i, td_j=td_j, depth=float(dj[0]) * 1.02))
    # the exact-(0,0,1) bearing branch of the tangent-base constructor (projectionTwoFrameOneCamFactor.cpp:36-38)
    c = dict(out[0]); c["pts_j"] = np.array([0.0, 0.0, 1.0]); out.append(c)
    return out


def ref_params(c):
    t = c["typ"]
    lam, td = np.array([c["lam"]]), np.array([c["td"]])
    if t == abi.PROJ_2F2C:
        return [c["pi"], c["pj"], c["ea"], c["eb"], lam, td]
    if t == abi.PROJ_1F2C:
        return [c["ea"], c["eb"], lam, td]
    return [c["pi"], c["pj"], c["ea"], lam, td]


def orc_proj(c):
    oc = tof.make_obs_const(c["pts_i"], c["pts_j"], c["vel_i"], c["vel_j"], c["td_i"], c["td_j"], depth=c["depth"])
    r, Ji, Jj, Ja, Jb, Jl, Jt = tof.proj_eval(c["typ"], oc, c["pi"], c["pj"], c["ea"], c["eb"], c["lam"], c["td"])
    t = c["typ"]
    if t == abi.PROJ_2F2C:
        Js = [Ji, Jj, Ja, Jb, Jl[:, None], Jt[:, None]]
    elif t == abi.PROJ_1F2C:
        Js = [Ja, Jb, Jl[:, None], Jt[:, None]]
    else:
        Js = [Ji, Jj, Ja, Jl[:, None], Jt[:, None]]
    return r, Js, np.array(oc.tangent_base).reshape(2, 3)


def imu_cases(seed=11, n=5):
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        steps = 20
        dt = np.full(steps, 0.005)
        acc = rng.normal(size=(steps + 1, 3)) * 0.5 + np.array([0, 0, 9.8]); gyr = rng.normal(size=(steps + 1, 3)) * 0.2
        ba0 = rng.normal(size=3) * 0.02; bg0 = rng.normal(size=3) * 0.003
        tof.RNG = np.random.default_rng(seed + 100 + k)
        pi = tof.rand_pose(0.5); pj = tof.plus(pi, np.concatenate([rng.normal(size=3) * 0.1, rng.normal(size=3) * 0.05]))
        sbi = np.concatenate([rng.normal(size=3), ba0 + rng.normal(size=3) * 0.01, bg0 + rng.normal(size=3) * 0.002])
        sbj = sbi + rng.normal(size=9) * 0.01
        out.append(dict(dt=dt, acc=acc, gyr=gyr, ba0=ba0, bg0=bg0, pi=pi, pj=pj, sbi=sbi, sbj=sbj))
    return out


def orc_imu(c):
    pre = orc.preintegrate(c["dt"], c["acc"], c["gyr"], c["ba0"], c["bg0"], 0.1, 0.05, 0.002, 0.0004)
    p = orc.OrcImuConst()
    p.sum_dt = pre["sum_dt"]; p.delta_p[:] = pre["delta_p"]; p.delta_q[:] = pre["delta_q"]; p.delta_v[:] = pre["delta_v"]
    p.linearized_ba[:] = c["ba0"]; p.linearized_bg[:] = c["bg0"]; p.jacobian[:] = pre["jacobian"]; p.covariance[:] = pre["covariance"]
    si = np.zeros(225)
    assert L.orc_imu_sqrt_info(abi.ptr(np.ascontiguousarray(pre["covariance"])), abi.ptr(si)) == 0
    p.sqrt_info[:] = si
    r = np.zeros(15); Js = [np.zeros((15, 7)), np.zeros((15, 9)), np.zeros((15, 7)), np.zeros((15, 9))]
    L.orc_imu_eval(C.byref(p), C.c_double(9.805), abi.ptr(c["pi"]), abi.ptr(c["sbi"]), abi.ptr(c["pj"]), abi.ptr(c["sbj"]), abi.ptr(r),
                   abi.ptr(Js[0]), abi.ptr(Js[1]), abi.ptr(Js[2]), abi.ptr(Js[3]))
    return pre, r, Js, si.reshape(15, 15)


def cons_cases(seed=13, n=6):
    rng = np.random.default_rng(seed)
    tof.RNG = np.random.default_rng(seed + 1)
    out = []
    for k in range(n):
        z = tof.rand_pose(1.0); x = tof.plus(z, np.concatenate([rng.normal(size=3) * 0.2, rng.normal(size=3) * 0.1]))
        if k == n - 1:
            x[3:7] = -x[3:7]      # other hemisphere: exercises positify inside Qleft (utils.hpp:56-63, 85-93)
        out.append(dict(z=z, x=x, tt=rng.normal(size=3) * 0.05, th=rng.normal(size=3) * 0.02, rho_T=10.0 ** rng.integers(0, 4), rho_theta=10.0 ** rng.integers(0, 4)))
    return out


def orc_cons(c):
    r = np.zeros(6); J = np.zeros((6, 7))
    L.orc_consensus_eval(abi.ptr(c["z"][:3].copy()), abi.ptr(c["z"][3:7].copy()), abi.ptr(c["tt"]), abi.ptr(c["th"]), C.c_double(c["rho_T"]), C.c_double(c["rho_theta"]),
                         abi.ptr(c["x"]), abi.ptr(r), abi.ptr(J))
    return r, J


# ----------------------------------------------------------------------------------------------- live reference vs oracle
def test_projection_factors_match_reference():
    g = None if HAVE_REF else frozen()
    worst = 0.0
    for i, c in enumerate(proj_cases()):
        if g is None:
            r_ref, J_ref, tb_ref = ref.proj_eval(c["typ"], c["pts_i"], c["pts_j"], c["vel_i"], c["vel_j"], c["td_i"], c["td_j"], c["depth"], ref_params(c))
        else:
            r_ref, J_ref, tb_ref = g[f"proj{i}_r"], [g[f"proj{i}_J{k}"] for k in range(len(ref_params(c)))], g[f"proj{i}_tb"]
        r_o, J_o, tb_o = orc_proj(c)
        close(tb_o, tb_ref, 1e-14)
        worst = max(worst, close(r_o, r_ref))
        for a, b in zip(J_o, J_ref):
            worst = max(worst, close(a, b))
    print("projection factors: worst scaled difference", worst)


PRE_FIELDS = ("sum_dt", "delta_p", "delta_q", "delta_v", "jacobian", "covariance")


def test_imu_factor_and_preintegration_match_reference():
    g = None if HAVE_REF else frozen()
    for i, c in enumerate(imu_cases()):
        pre_o, r_o, J_o, si_o = orc_imu(c)
        if g is None:
            pre_r = ref.preintegrate(c["dt"], c["acc"], c["gyr"], c["ba0"], c["bg0"])
            r_r, J_r, si_r = ref.imu_eval(pre_r, c["ba0"], c["bg0"], c["pi"], c["sbi"], c["pj"], c["sbj"])
        else:
            pre_r = {k: g[f"imu{i}_pre_{k}"] for k in PRE_FIELDS}
            r_r, J_r, si_r = g[f"imu{i}_r"], [g[f"imu{i}_J{k}"] for k in range(4)], g[f"imu{i}_sqrt_info"]
        for k in PRE_FIELDS:
            close(np.ravel(pre_o[k]), np.ravel(pre_r[k]), 1e-13)
        # sqrt_info = LLT(cov^-1).L^T: conditioning of cov (1e8) bounds the agreement of two different inversion routes
        close(si_o, si_r, 1e-8)
        close(r_o, r_r, 1e-8)
        for a, b in zip(J_o, J_r):
            close(a, b, 1e-8)
        # with the reference's own sqrt_info the restated raw residual / Jacobians agree to rounding
        Ui = np.linalg.inv(si_r)
        close(np.linalg.solve(si_o, r_o), Ui @ r_r, 1e-11)
        for a, b in zip(J_o, J_r):
            close(np.linalg.solve(si_o, a), Ui @ b, 1e-11)


def test_consensus_factor_matches_reference():
    g = None if HAVE_REF else frozen()
    for i, c in enumerate(cons_cases()):
        if g is None:
            r_r, J_r = ref.consensus_eval(c["z"][:3], c["z"][3:7], c["tt"], c["th"], c["rho_T"], c["rho_theta"], c["x"])
        else:
            r_r, J_r = g[f"cons{i}_r"], g[f"cons{i}_J"]
        r_o, J_o = orc_cons(c)
        close(r_o, r_r, 1e-14); close(J_o, J_r, 1e-14)


def manifold_cases():
    rng = np.random.default_rng(17)
    tof.RNG = np.random.default_rng(18)
    plus = [(tof.rand_pose(2.0), rng.normal(size=6) * 0.3) for _ in range(8)]
    x_jac = tof.rand_pose()
    qs = np.array([tof.rand_pose()[3:7] for _ in range(5)])
    qs[1:] = qs[0] + 0.05 * qs[1:]; qs /= np.linalg.norm(qs, axis=1, keepdims=True)
    return plus, x_jac, qs


def reference_manifold(plus, x_jac, qs):
    """PoseLocalParameterization::Plus on every (x, delta), its ComputeJacobian at x_jac, the average of qs."""
    return np.array([ref.pose_plus(x, d) for x, d in plus]), ref.pose_plus_jacobian(x_jac), ref.average_quats(qs)


def test_manifold_and_quaternion_helpers_match_reference():
    plus, x_jac, qs = manifold_cases()
    if HAVE_REF:
        plus_r, J, a_r = reference_manifold(plus, x_jac, qs)
    else:
        g = frozen()
        plus_r, J, a_r = g["manifold_plus"], g["manifold_plus_jacobian"], g["manifold_average_quat"]
    for (x, d), p_r in zip(plus, plus_r):
        o = np.zeros(7)
        L.orc_pose_plus(abi.ptr(x), abi.ptr(d), abi.ptr(o))
        close(o, p_r, 1e-15)
        close(synth.pose_plus(x, d), p_r, 1e-15)
    assert np.array_equal(J, np.vstack([np.eye(6), np.zeros((1, 6))]))     # pose_local_parameterization.cpp:31-38
    a_o = np.zeros(4)
    L.orc_average_quats(C.c_int(len(qs)), abi.ptr(qs), abi.ptr(a_o))
    assert min(np.abs(a_r - a_o).max(), np.abs(a_r + a_o).max()) <= 1e-12      # eigenvector sign is free


# ----------------------------------------------------------------------------------------------- marginalization prior
def prior_cases(seed=41):
    rng = np.random.default_rng(seed)
    tof.RNG = np.random.default_rng(seed + 1)
    out = []
    for case in range(4):
        kinds = [[0, 2], [0, 2, 1, 3, 4, 0], [0, 2, 0, 2, 4, 4, 4], [1, 0, 2]][case]
        x0, x = [], []
        for k in kinds:
            if k in (0, 1):
                p0 = tof.rand_pose(2.0); x0.append(p0)
                p1 = tof.plus(p0, np.concatenate([rng.normal(size=3) * 0.1, rng.normal(size=3) * 0.05]))
                if case == 3 and k == 0:
                    p1[3:7] = -p1[3:7]            # other hemisphere: the `!(qerr.w() >= 0)` branch (prior_factor.cpp:64-66)
                x.append(p1)
            else:
                v = rng.normal(size=ref.PRIOR_SIZE[k]); x0.append(v); x.append(v + 0.05 * rng.normal(size=ref.PRIOR_SIZE[k]))
        m = sum(ref.PRIOR_EFF[k] for k in kinds)
        M = rng.normal(size=(m - (3 if case % 2 else 0), m))                     # odd cases: rank deficient (eigenvalue clamp)
        out.append(dict(kinds=np.array(kinds, np.int32), x0=np.concatenate(x0), x=np.concatenate(x), A=M.T @ M, b=rng.normal(size=m)))
    return out


def orc_prior(c):
    m = len(c["b"]); J = np.zeros((m, m)); e0 = np.zeros(m)
    L.orc_to_jac_res(C.c_int(m), abi.ptr(c["A"]), abi.ptr(c["b"]), abi.ptr(J), abi.ptr(e0))
    dx = np.zeros(m); off = eo = 0
    for k in c["kinds"]:
        sz, ef = ref.PRIOR_SIZE[k], ref.PRIOR_EFF[k]
        if k in (0, 1):
            d = np.zeros(6); L.orc_prior_dx_pose(abi.ptr(c["x"][off:off + 7].copy()), abi.ptr(c["x0"][off:off + 7].copy()), abi.ptr(d)); dx[eo:eo + 6] = d
        else:
            dx[eo:eo + ef] = c["x"][off:off + sz] - c["x0"][off:off + sz]
        off += sz; eo += ef
    return e0 + J @ dx, J                                                        # orc_solver.c:495-512


def check_prior(c, r_ref, J_ref):
    r_o, J_o = orc_prior(c)
    # the rows of (J, e0) are eigenvectors scaled by sqrt(eigenvalue): their sign is the eigen-solver's choice -- compare what
    # enters the normal equations, and the rows themselves up to sign
    close(J_o.T @ J_o, J_ref.T @ J_ref, 1e-12); close(J_o.T @ r_o, J_ref.T @ r_ref, 1e-12); close(r_o @ r_o, r_ref @ r_ref, 1e-12)
    sg = np.sign(np.sum(J_o * J_ref, axis=1)); sg[sg == 0] = 1.0
    close(J_o, J_ref * sg[:, None], 1e-11); close(r_o, r_ref * sg, 1e-11)


def test_prior_factor_matches_reference():
    """orc_to_jac_res + orc_prior_dx_pose + `r = e0 + J dx` (the oracle's prior) vs the reference's PriorFactor built from the
    same information form (A, b): toJacRes (eigenvalue clamp at 1e-8, rank-deficient cases) and Evaluate (pose dx with the
    hemisphere branch, Euclidean blocks), prior_factor.cpp:45-90, :132-177 compiled unmodified.  (The eigen-decomposition
    under the reference code is the shim's cyclic-Jacobi stand-in of Eigen::SelfAdjointEigenSolver.)"""
    g = None if HAVE_REF else frozen()
    for i, c in enumerate(prior_cases()):
        check_prior(c, *(ref.prior_eval(c["kinds"], c["x0"], c["x"], c["A"], c["b"]) if g is None else (g[f"prior{i}_r"], g[f"prior{i}_J"])))


# ----------------------------------------------------------------------------------------------- marginalization
MARG_CASES = [dict(seed=9, n_landmarks=40, n_frames=5), dict(seed=10, n_landmarks=30, n_frames=4, cams="stereo"),
              dict(seed=12, n_landmarks=30, n_frames=4, cams="stereo", estimate_extrinsic=True, estimate_td=True, td_offset=0.002)]
_EFF = {0: 6, 1: 6, 2: 9, 3: 1, 4: 1}


def _offsets(refs):
    off, o_ = {}, 0
    for r in refs:
        off[(int(r["kind"]), int(r["id"]))] = (o_, _EFF[int(r["kind"])]); o_ += _EFF[int(r["kind"])]
    return off


def check_marginalization(kw, refs_r, x0_r, J_r, e0_r):
    pr = synth.make_window(**kw)
    o = orc.Oracle(); pr.load(o)
    A, b, refs, x0 = o.marginalize([int(pr["frame_ids"][0])])
    oo, ro = _offsets(refs), _offsets(refs_r)
    assert set(oo) == set(ro)                                     # the same blocks are kept
    perm = np.concatenate([np.arange(ro[k][0], ro[k][0] + ro[k][1]) for k in oo])
    # the reference hands the new prior over as (J, e0) = toJacRes(A, b): J^T J = A and J^T e0 = b on the kept eigen-space
    close(A, (J_r.T @ J_r)[np.ix_(perm, perm)], 1e-9); close(b, (J_r.T @ e0_r)[perm], 1e-9)
    # linearisation points of the kept blocks = their current values, in the reference's block order
    SIZE = {0: 7, 1: 7, 2: 9, 3: 1, 4: 1}
    xo, xr, a, c = {}, {}, 0, 0
    for r in refs:
        k = (int(r["kind"]), int(r["id"])); xo[k] = x0[a:a + SIZE[k[0]]]; a += SIZE[k[0]]
    for r in refs_r:
        k = (int(r["kind"]), int(r["id"])); xr[k] = x0_r[c:c + SIZE[k[0]]]; c += SIZE[k[0]]
    for k in xo:
        close(xo[k], xr[k], 1e-15)


def test_marginalization_matches_the_reference_marginalizer():
    """orc_marginalize_x0 vs the reference's OWN Marginalizer::marginalize (marginalization.cpp, ParamResidualInfo.{hpp,cpp},
    BaseParamResInfo.cpp, utils.hpp schurComplement, PriorFactor -- compiled unmodified) run over the reference's factor
    objects of the same window with Huber(1): same kept blocks, A and b of the new prior, linearisation points.  Mono, stereo
    (2F2C / 1F2C residual infos) and free-extrinsic / td windows; first frame removed, remove_base_when_margin_remote = 2,
    FEJ off, sparse-LLT Schur complement (config/tum/tum_single.yaml:87-94)."""
    if not HAVE_REF:
        g = frozen()
        for i, kw in enumerate(MARG_CASES):
            check_marginalization(kw, g[f"marg{i}_refs"], g[f"marg{i}_x0"], g[f"marg{i}_J"], g[f"marg{i}_e0"])
        return
    ref.configure()
    for kw in MARG_CASES:
        pr = synth.make_window(**kw)
        check_marginalization(kw, *ref.marginalize(pr, [int(pr["frame_ids"][0])]))


# ----------------------------------------------------------------------------------------------- ADMM loop
ADMM_KW = dict(rho_frame_T=30.0, rho_frame_theta=70.0, relaxation_alpha=0.6)
ADMM_STEPS, ADMM_ITERS_PER_STEP = 4, 2


def admm_trajectory():
    """The oracle's ADMM (orc_admm_solve) run for 0, 1, .. K consensus steps from the same start (each run is a prefix of the
    next: fixed iterations per step) -> per run and agent: consensus slots, local poses, z, tilde."""
    sw = synth.make_swarm(seed=5, n_agents=3, n_frames=4, n_landmarks=40, shared_per_pair=15)
    runs = []
    for k in range(ADMM_STEPS + 1):
        ags = []
        for p in sw:
            o = orc.Oracle(max_num_iterations=ADMM_ITERS_PER_STEP * max(k, 1), consensus_max_steps=max(k, 1), **ADMM_KW); p.load(o); ags.append(o)
        if k:
            orc.admm_solve(ags, fixed_mode=True)
        out = []
        for p, o in zip(sw, ags):
            refs, slots, _ = p["consensus"]
            x = np.array([o.get_blocks(int(r["kind"]), [int(r["id"])])[0] for r in refs])
            z, t = o.get_consensus(refs)
            out.append((slots, x, z, t))
        runs.append(out)
    n_slots = sw[0]["consensus"][2]
    present = np.zeros((len(sw), n_slots), np.uint8); traj = np.zeros((ADMM_STEPS + 1, len(sw), n_slots, 7)); traj[..., 6] = 1.0
    for k, out in enumerate(runs):
        for a, (slots, x, _, _) in enumerate(out):
            present[a, slots] = 1; traj[k, a, slots] = x
    return runs, present, traj


def check_admm(runs, traj, z, tl, rs):
    for k in range(1, ADMM_STEPS + 1):
        for a, (slots, _, z_o, t_o) in enumerate(runs[k]):
            z_r, t_r = z[k - 1, a, slots], tl[k - 1, a, slots]
            sgn = np.sign(np.sum(z_r[:, 3:] * z_o[:, 3:], axis=1, keepdims=True))     # the averaged quaternion's sign is free
            close(z_o[:, :3], z_r[:, :3], 1e-13); close(z_o[:, 3:], z_r[:, 3:] * sgn, 1e-13)
            close(t_o, t_r, 1e-13)
            # the ConsenusPoseFactor objects the reference loop created (argument order of rho / tilde segments included),
            # evaluated at the step's local poses, vs the oracle's factor with the oracle's z / tilde
            for i, s_ in enumerate(slots):
                c = dict(z=z_o[i], x=traj[k - 1, a, s_], tt=t_o[i, :3].copy(), th=t_o[i, 3:].copy(), rho_T=ADMM_KW["rho_frame_T"], rho_theta=ADMM_KW["rho_frame_theta"])
                close(orc_cons(c)[0], rs[k - 1, a, s_], 1e-12)


def test_admm_bookkeeping_matches_the_reference_loop():
    """The reference's own ConsensusSolver::solve loop (ConsensusSolver.cpp:39-235, compiled unmodified; syncData /
    updateGlobal / updateTilde, 3 agents on 3 threads, relaxation 0.6) replays the oracle's trajectory of local poses: global
    averages z, duals tilde and the created consensus factors must equal the oracle's at every step."""
    runs, present, traj = admm_trajectory()
    if HAVE_REF:
        z, tl, rs = ref.admm_replay(present, traj, ADMM_KW["relaxation_alpha"], ADMM_KW["rho_frame_T"], ADMM_KW["rho_frame_theta"])
    else:
        g = frozen()
        z, tl, rs = g["admm_z"], g["admm_tilde"], g["admm_res"]
    assert np.abs(tl[-1]).max() > 1e-3      # the duals are not trivially zero
    check_admm(runs, traj, z, tl, rs)


# ----------------------------------------------------------------------------------------------- loss corrector
def loss_cases(seed=31):
    rng = np.random.default_rng(seed)
    out = []
    for k in range(8):
        n = 2 + (k % 2)                                  # reprojection (2) and depth-augmented (3) residual blocks
        out.append(dict(r=rng.normal(size=n) * (0.3 if k < 3 else 4.0), J=rng.normal(size=(n, 7)), a=1.0 if k % 4 else 0.5))
    out.append(dict(r=np.zeros(2), J=rng.normal(size=(2, 7)), a=1.0))   # sq_norm == 0 branch
    return out


def orc_loss(c):
    r, J = c["r"], c["J"]
    rho = np.zeros(3); s = float(r @ r)
    L.orc_huber(C.c_double(c["a"]), C.c_double(s), abi.ptr(rho))
    rs = C.c_double(); sr = C.c_double(); asn = C.c_double()
    L.orc_corrector(abi.ptr(rho), C.c_double(s), C.byref(rs), C.byref(sr), C.byref(asn))
    return rs.value * r, sr.value * (J - asn.value * np.outer(r, r @ J))     # orc_solver.c:435-452


def test_loss_corrector_matches_reference():
    """orc_huber + orc_corrector as the oracle's minimiser applies them vs the reference's ResidualInfo::Evaluate loss section
    (d2common/src/solver/BaseParamResInfo.cpp:71-92, compiled unmodified) with ceres::HuberLoss(a)."""
    g = None if HAVE_REF else frozen()
    for i, c in enumerate(loss_cases()):
        r_r, J_r = ref.loss_correct(c["r"], c["J"], c["a"]) if g is None else (g[f"loss{i}_r"], g[f"loss{i}_J"])
        r_o, J_o = orc_loss(c)
        close(r_o, r_r, 1e-15); close(J_o, J_r, 1e-15)


# ----------------------------------------------------------------------------------------------- pose-graph factor (d2pgo)
def relpose_cases(seed=23, n=8):
    rng = np.random.default_rng(seed)
    tof.RNG = np.random.default_rng(seed + 1)
    out = []
    for k in range(n):
        pa, pb = tof.rand_pose(3.0), tof.rand_pose(3.0)
        rel = tof.rand_pose(2.0)
        S = np.diag([20.0, 20.0, 20.0, 57.0, 57.0, 57.0]) + (0.0 if k % 2 == 0 else 1.0) * rng.normal(size=(6, 6))   # diagonal and full
        out.append(dict(pa=pa, pb=pb, rel=rel, S=S))
    return out


def plus_jacobian(x):
    """d (x (+) delta) / d delta at 0 for PoseLocalParameterization::Plus (pose_local_parameterization.cpp:13-29): 7 x 6.
    (The class's own ComputeJacobian is the VINS-style [I6; 0] placeholder, not this derivative.)"""
    v, w = x[3:6], x[6]
    P = np.zeros((7, 6)); P[:3, :3] = np.eye(3)
    P[3:6, 3:] = 0.5 * (w * np.eye(3) + np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])); P[6, 3:] = -0.5 * v
    return P


def check_relpose(c, r_ref, Ja, Jb):
    from oracle import pgo_oracle as po
    r_o, J0, J1 = po.edge_eval(c["pa"], c["pb"], c["rel"], c["S"])
    close(r_o, r_ref, 1e-13)
    # the reference Jacobians are w.r.t. the 7 ambient parameters (what autodiff hands to the manifold); the oracle's and the
    # device's are in the tangent of the right-multiplicative retraction: J_tangent = J_ambient d(x (+) delta)/d delta
    close(J0, Ja @ plus_jacobian(c["pa"]), 1e-13); close(J1, Jb @ plus_jacobian(c["pb"]), 1e-13)


def test_rel_pose_factor_matches_reference():
    """oracle/pgo_oracle.py::edge_eval vs the reference's RelPoseFactorAD functor (RelPoseFactor.hpp:68-135) run with doubles
    (residual) and with dual numbers (exact derivatives of the reference's own residual code)."""
    g = None if HAVE_REF else frozen()
    for i, c in enumerate(relpose_cases()):
        check_relpose(c, *(ref.relpose_ad_eval(c["pa"], c["pb"], c["rel"], c["S"]) if g is None else (g[f"relpose{i}_r"], g[f"relpose{i}_Ja"], g[f"relpose{i}_Jb"])))


def relpose4d_cases(seed=29, n=8):
    rng = np.random.default_rng(seed)
    tof.RNG = np.random.default_rng(seed + 1)
    out = []
    for k in range(n):
        pa = np.concatenate([rng.normal(size=3) * 3, [rng.uniform(-np.pi, np.pi)]]); pb = np.concatenate([rng.normal(size=3) * 3, [rng.uniform(-np.pi, np.pi)]])
        if k == n - 1:
            pa[3], pb[3] = 3.0, -3.0                      # yaw difference wraps through pi
        S = np.diag([20.0, 20.0, 20.0, 57.0]) + (0.0 if k % 2 == 0 else 1.0) * rng.normal(size=(4, 4))
        out.append(dict(pa=pa, pb=pb, rel=tof.rand_pose(2.0), S=S))
    return out


def check_relpose4d(c, r_ref, Ja, Jb):
    from oracle import pgo_oracle as po
    q = c["rel"][3:7]
    yaw = np.arctan2(2 * (q[3] * q[2] + q[0] * q[1]), 1 - 2 * (q[1] * q[1] + q[2] * q[2]))      # Swarm::Pose::yaw (ASSUMED: the z Euler angle)
    r_o, J0, J1 = po.edge_eval_4d(c["pa"], c["pb"], c["rel"][:3], yaw, c["S"])
    close(r_o, r_ref, 1e-13); close(J0, Ja, 1e-13); close(J1, Jb, 1e-13)


def test_rel_pose_factor_4d_matches_reference():
    """oracle/pgo_oracle.py::edge_eval_4d vs the reference's RelPoseFactor4D functor (RelPoseFactor.hpp:196-238; d2pgo's default
    4-DoF configuration) with doubles and dual numbers.  Oracle-level only: the device path carries the 6-DoF factor."""
    g = None if HAVE_REF else frozen()
    for i, c in enumerate(relpose4d_cases()):
        check_relpose4d(c, *(ref.relpose4d_eval(c["pa"], c["pb"], c["rel"], c["S"]) if g is None else (g[f"relpose4d{i}_r"], g[f"relpose4d{i}_Ja"], g[f"relpose4d{i}_Jb"])))


# ----------------------------------------------------------------------------------------------- frozen reference outputs
def test_oracle_matches_golden_reference_vectors():
    """Same comparisons against reference outputs frozen by tests/golden/make_ref_golden.py (runs everywhere)."""
    g = np.load(GOLD)
    for i, c in enumerate(proj_cases()):
        r_o, J_o, tb_o = orc_proj(c)
        close(r_o, g[f"proj{i}_r"]); close(tb_o, g[f"proj{i}_tb"], 1e-14)
        for k, a in enumerate(J_o):
            close(a, g[f"proj{i}_J{k}"])
    for i, c in enumerate(imu_cases()):
        pre_o, r_o, J_o, si_o = orc_imu(c)
        close(np.ravel(pre_o["jacobian"]), g[f"imu{i}_pre_jacobian"], 1e-13); close(np.ravel(pre_o["covariance"]), g[f"imu{i}_pre_covariance"], 1e-13)
        close(si_o, g[f"imu{i}_sqrt_info"], 1e-8); close(r_o, g[f"imu{i}_r"], 1e-8)
        for k, a in enumerate(J_o):
            close(a, g[f"imu{i}_J{k}"], 1e-8)
    for i, c in enumerate(cons_cases()):
        r_o, J_o = orc_cons(c)
        close(r_o, g[f"cons{i}_r"], 1e-14); close(J_o, g[f"cons{i}_J"], 1e-14)
    for i, c in enumerate(relpose_cases()):
        check_relpose(c, g[f"relpose{i}_r"], g[f"relpose{i}_Ja"], g[f"relpose{i}_Jb"])
    for i, c in enumerate(loss_cases()):
        r_o, J_o = orc_loss(c)
        close(r_o, g[f"loss{i}_r"], 1e-15); close(J_o, g[f"loss{i}_J"], 1e-15)
    runs, _, traj = admm_trajectory()
    check_admm(runs, traj, g["admm_z"], g["admm_tilde"], g["admm_res"])
    for i, c in enumerate(prior_cases()):
        check_prior(c, g[f"prior{i}_r"], g[f"prior{i}_J"])
    for i, kw in enumerate(MARG_CASES):
        check_marginalization(kw, g[f"marg{i}_refs"], g[f"marg{i}_x0"], g[f"marg{i}_J"], g[f"marg{i}_e0"])
    for i, c in enumerate(relpose4d_cases()):
        check_relpose4d(c, g[f"relpose4d{i}_r"], g[f"relpose4d{i}_Ja"], g[f"relpose4d{i}_Jb"])
