"""Pose-graph path (include/d2pgo.h, BASELINE config 5 / SURVEY 8f rank 3): factor restatement vs finite differences,
g2o round trip in the reference's multi-agent id convention, edge sharding == full product (gloo-free numpy check),
and on the GPU: per-edge residual / Jacobians and the converged solution against the scipy oracle."""
import os

import numpy as np
import pytest

from d2slam_b200 import pgo, synth
from oracle import pgo_oracle as po

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_extra.npz")


def small_graph(seed=1, n_agents=3, n=40, loops=120):
    return pgo.make_pose_graph(seed=seed, n_agents=n_agents, poses_per_agent=n, loops=loops)


def test_rel_pose_factor_restatement_matches_finite_differences():
    rng = np.random.default_rng(3)
    g = small_graph()
    S = g["sqrt_info"].reshape(-1, 6, 6)
    for e in rng.integers(0, len(g["ea"]), 10):
        a, b = g["ea"][e], g["eb"][e]
        p0, p1 = g["init"][a], g["init"][b]
        r, J0, J1 = po.edge_eval(p0, p1, g["rel"][e], S[e])
        eps = 1e-6
        for J, which in ((J0, 0), (J1, 1)):
            num = np.zeros((6, 6))
            for k in range(6):
                d = np.zeros(6); d[k] = eps
                pp = [p0, p1]; pm = [p0, p1]
                pp[which] = synth.pose_plus(pp[which], d); pm[which] = synth.pose_plus(pm[which], -d)
                num[:, k] = (po.edge_eval(pp[0], pp[1], g["rel"][e], S[e])[0] - po.edge_eval(pm[0], pm[1], g["rel"][e], S[e])[0]) / (2 * eps)
            assert np.abs(num - J).max() <= 1e-6 * max(1.0, np.abs(J).max()), (which, np.abs(num - J).max())


def test_g2o_round_trip_multi_agent_ids(tmp_path):
    g = small_graph(seed=2, n_agents=3, n=12, loops=20)
    path = str(tmp_path / "graph.g2o")
    pgo.write_g2o(path, g["ids"], g["init"], g["id_a"], g["id_b"], g["rel"], g["sqrt_info"])
    assert pgo.g2o_split_id(pgo.g2o_vertex_id(2, 77)) == (2, 77) and pgo.g2o_split_id(123) == (0, 123)
    h = pgo.read_g2o(path)
    assert np.array_equal(h["ids"], g["ids"]) and np.array_equal(h["id_a"], g["id_a"]) and np.array_equal(h["id_b"], g["id_b"])
    assert np.allclose(h["poses"], g["init"], atol=1e-15) and np.allclose(h["rel"], g["rel"], atol=1e-15)
    S0 = g["sqrt_info"].reshape(-1, 6, 6); S1 = h["sqrt_info"].reshape(-1, 6, 6)
    assert np.allclose(np.einsum("eij,eik->ejk", S1, S1), np.einsum("eij,eik->ejk", S0, S0), rtol=1e-12)
    only0 = pgo.read_g2o(path, max_agent_id=0)
    assert set(only0["ids"] // 1_000_000) == {0} and len(only0["id_a"]) < len(h["id_a"])


def test_edge_sharding_sums_to_the_full_normal_equations():
    """What the multi-GPU path relies on: J^T J p summed over edge shards (e % nranks) == the full product."""
    g = small_graph(seed=4)
    S = g["sqrt_info"].reshape(-1, 6, 6); N = len(g["ids"])
    rng = np.random.default_rng(0); p = rng.normal(size=(N, 6))

    def product(sel):
        y = np.zeros((N, 6))
        for e in sel:
            a, b = g["ea"][e], g["eb"][e]
            _, J0, J1 = po.edge_eval(g["init"][a], g["init"][b], g["rel"][e], S[e])
            t = J0 @ p[a] + J1 @ p[b]; y[a] += J0.T @ t; y[b] += J1.T @ t
        return y
    E = len(g["ea"]); full = product(range(E))
    parts = sum(product(range(r, E, 3)) for r in range(3))
    assert np.abs(full - parts).max() <= 1e-9 * np.abs(full).max()


@pytest.mark.gpu
def test_pgo_edges_on_device_match_oracle():
    g = small_graph(seed=5)
    s = pgo.PgoSolver()
    s.set_poses(g["ids"], g["init"], g["fixed"]); s.add_edges(g["id_a"], g["id_b"], g["rel"], g["sqrt_info"])
    dev = s.debug_edges()
    S = g["sqrt_info"].reshape(-1, 6, 6)
    for e in range(0, len(dev), 7):
        r, J0, J1 = po.edge_eval(g["init"][g["ea"][e]], g["init"][g["eb"][e]], g["rel"][e], S[e])
        ref = np.concatenate([r, J0.ravel(), J1.ravel()])
        assert np.abs(dev[e] - ref).max() <= 1e-11 * max(1.0, np.abs(ref).max())


@pytest.mark.gpu
def test_pgo_converged_solution_matches_sparse_direct_oracle():
    g = small_graph(seed=6, n_agents=4, n=60, loops=300)
    s = pgo.PgoSolver(max_iterations=40, pcg_max_iterations=400, pcg_tolerance=1e-12, lambda0=0.0, function_tolerance=1e-14)
    s.set_poses(g["ids"], g["init"], g["fixed"]); s.add_edges(g["id_a"], g["id_b"], g["rel"], g["sqrt_info"])
    rep = s.solve()
    x_ref, costs = po.solve(g["init"], g["fixed"], g["ea"], g["eb"], g["rel"], g["sqrt_info"], iters=40)
    assert rep.final_cost < rep.initial_cost and abs(rep.final_cost - costs[-1]) <= 1e-8 * costs[-1], (rep.final_cost, costs[-1])
    dp, dr = synth.pose_errors(s.get_poses(g["ids"]), x_ref)
    assert dp <= 1e-6 and dr <= 1e-6, (dp, dr)
    # and it actually removed the drift: far closer to the ground truth than the initial guess
    e0, _ = synth.pose_errors(g["init"], g["gt"]); e1, _ = synth.pose_errors(s.get_poses(g["ids"]), g["gt"])
    assert e1 < 0.5 * e0


def functor_case():
    """Graph, full square-root information matrices and the edges compared with the reference's RelPoseFactorAD functor."""
    g = small_graph(seed=8)
    rng = np.random.default_rng(1)
    S = g["sqrt_info"].reshape(-1, 6, 6) + 0.5 * rng.normal(size=(len(g["ea"]), 6, 6))      # full square-root information
    return g, S, np.arange(0, len(g["ea"]), 5)


def reference_functor(g, S, edges):
    """RelPoseFactorAD on `edges` (oracle/_ref/libd2ref.so: doubles for the residual, dual numbers for the exact ambient
    Jacobians) -> residuals [n, 6], Jacobians [n, 6, 7] of pose a and of pose b."""
    from oracle import ref
    out = [ref.relpose_ad_eval(g["init"][g["ea"][e]], g["init"][g["eb"][e]], g["rel"][e], S[e]) for e in edges]
    return tuple(np.array(x) for x in zip(*out))


def reference_answers(key):
    """None where the reference library is present (the caller runs it); else the answers it gave on the same seeded inputs,
    frozen in tests/golden/ref_extra.npz by tests/golden/make_ref_golden.py."""
    from oracle import ref
    if ref.available():
        return None
    g = np.load(GOLD)
    return {k[len(key) + 1:]: g[k] for k in g.files if k.startswith(key + "_")}


@pytest.mark.gpu
def test_pgo_edges_on_device_match_the_reference_functor():
    """Device residual / tangent Jacobians of every sampled edge vs the reference's own RelPoseFactorAD functor."""
    from test_ref_pin import plus_jacobian
    g, S, edges = functor_case()
    s = pgo.PgoSolver()
    s.set_poses(g["ids"], g["init"], g["fixed"]); s.add_edges(g["id_a"], g["id_b"], g["rel"], S.reshape(-1, 36))
    dev = s.debug_edges()
    frozen = reference_answers("functor")
    r, Ja, Jb = reference_functor(g, S, edges) if frozen is None else (frozen["r"], frozen["Ja"], frozen["Jb"])
    for n, e in enumerate(edges):
        a, b = g["ea"][e], g["eb"][e]
        want = np.concatenate([r[n], (Ja[n] @ plus_jacobian(g["init"][a])).ravel(), (Jb[n] @ plus_jacobian(g["init"][b])).ravel()])
        assert np.abs(dev[e] - want).max() <= 1e-11 * max(1.0, np.abs(want).max()), e


def g2o_agents_case(directory):
    """The multi-agent graph written by pgo.write_g2o_agents into `directory` -> (graph, information matrices, agents)."""
    g = small_graph(seed=2, n_agents=3, n=12, loops=20)
    rng = np.random.default_rng(0)
    S = g["sqrt_info"].reshape(-1, 6, 6) + 0.3 * rng.normal(size=(len(g["ea"]), 6, 6))        # full information matrices
    info = np.einsum("eki,ekj->eij", S, S)
    agents = pgo.write_g2o_agents(directory, g["ids"], g["init"], g["id_a"], g["id_b"], g["rel"], S.reshape(-1, 36))
    return g, info, agents


G2O_READ_FIELDS = ("v_agent", "v_id", "v_pose", "e_agent_a", "e_id_a", "e_agent_b", "e_id_b", "e_rel", "e_info")


def reference_g2o_reads(directory, agents):
    """read_g2o_agent on every agent's file, with all agents and with max_agent_id = 0 -> {name: array}."""
    from oracle import ref
    out = {}
    for a in agents:
        path = os.path.join(directory, f"{a}.g2o")
        r = ref.g2o_read(path, max_agent_id=len(agents) - 1)
        out.update({f"{a}_{k}": r[k] for k in G2O_READ_FIELDS})
        r0 = ref.g2o_read(path, max_agent_id=0)
        out[f"{a}_only0_counts"] = np.array([len(r0["v_id"]), len(r0["e_id_a"])])
        with open(path, "rb") as f:
            out[f"{a}_file"] = np.frombuffer(f.read(), np.uint8)
    return out


def test_g2o_written_here_is_read_by_the_reference_reader(tmp_path):
    """pgo.write_g2o_agents (one `<agent>.g2o` per agent, chr('a' + agent) in the top byte of every vertex id) -> the reference's
    OWN read_g2o_agent (d2pgo/test/posegraph_g2o.cpp, compiled unmodified into oracle/_ref) on every file: agents, keyframe ids,
    poses, relative poses and information matrices come back exactly; the max_agent_id filter drops the same edges as ours.
    Without the library: its answers on byte-identical files."""
    g, info, agents = g2o_agents_case(str(tmp_path))
    assert agents == [0, 1, 2]
    reads = reference_answers("g2o_agents")
    if reads is None:
        reads = reference_g2o_reads(str(tmp_path), agents)
    for a in agents:
        with open(tmp_path / f"{a}.g2o", "rb") as f:
            assert np.array_equal(np.frombuffer(f.read(), np.uint8), reads[f"{a}_file"])      # the files the answers are about
        r = {k: reads[f"{a}_{k}"] for k in G2O_READ_FIELDS}
        v = (g["ids"] // 1_000_000) == a; e = (g["id_a"] // 1_000_000) == a
        assert np.all(r["v_agent"] == a) and np.array_equal(np.sort(r["v_id"]), np.sort(g["ids"][v] % 1_000_000))
        order = np.argsort(r["v_id"]); mine = np.argsort(g["ids"][v])
        assert np.abs(r["v_pose"][order] - g["init"][v][mine]).max() <= 1e-15
        assert np.array_equal(r["e_agent_a"].astype(np.int64) * 1_000_000 + r["e_id_a"], g["id_a"][e])
        assert np.array_equal(r["e_agent_b"].astype(np.int64) * 1_000_000 + r["e_id_b"], g["id_b"][e])
        assert np.abs(r["e_rel"] - g["rel"][e]).max() <= 1e-15
        assert np.abs(r["e_info"] - info[e]).max() <= 1e-12 * np.abs(info).max()
        # the agent filter (posegraph_g2o.cpp:72-74, 112-114): with max_agent_id = 0 only agent 0's own edges survive
        m0 = pgo.read_g2o(str(tmp_path / f"{a}.g2o"), max_agent_id=0)
        assert np.array_equal(reads[f"{a}_only0_counts"], [len(m0["ids"]), len(m0["id_a"])])
    h = pgo.read_g2o_agents(str(tmp_path), 3)
    assert np.array_equal(np.sort(h["ids"]), np.sort(g["ids"])) and len(h["id_a"]) == len(g["id_a"])
    h2 = pgo.read_g2o_agents(str(tmp_path), 2)
    assert set(h2["ids"] // 1_000_000) == {0, 1} and np.all(h2["id_b"] // 1_000_000 <= 1)


def reference_written_case():
    g = small_graph(seed=3, n_agents=1, n=15, loops=10)
    S = g["sqrt_info"].reshape(-1, 6, 6)
    return g, np.einsum("eki,ekj->eij", S, S)


def reference_g2o_write(path, g, info):
    from oracle import ref
    ref.g2o_write(path, g["ids"], g["init"], g["id_a"], g["id_b"], g["rel"], info)


def test_g2o_written_by_the_reference_is_read_here(tmp_path):
    """The reference's write_result_to_g2o (plain keyframe ids, default ostream precision: 6 significant digits) -> pgo.read_g2o.
    Without the library: the file it wrote for the same graph."""
    g, info = reference_written_case()
    path = str(tmp_path / "out.g2o")
    frozen = reference_answers("g2o_written")
    if frozen is None:
        reference_g2o_write(path, g, info)
    else:
        with open(path, "wb") as f:
            f.write(frozen["file"].tobytes())
    h = pgo.read_g2o(path)
    assert np.array_equal(h["ids"], g["ids"]) and np.array_equal(h["id_a"], g["id_a"]) and np.array_equal(h["id_b"], g["id_b"])
    assert np.abs(h["poses"][:, :3] - g["init"][:, :3]).max() <= 1e-5 * max(1.0, np.abs(g["init"][:, :3]).max()) and np.abs(h["poses"][:, 3:] - g["init"][:, 3:]).max() <= 1e-5
    assert np.abs(h["rel"] - g["rel"]).max() <= 1e-5 * max(1.0, np.abs(g["rel"]).max())
    S1 = h["sqrt_info"].reshape(-1, 6, 6)
    assert np.abs(np.einsum("eki,ekj->eij", S1, S1) - info).max() <= 1e-5 * np.abs(info).max()


def test_batched_linearisation_equals_the_per_edge_function():
    g = small_graph(seed=7)
    rng = np.random.default_rng(2)
    S = g["sqrt_info"].reshape(-1, 6, 6) + 0.4 * rng.normal(size=(len(g["ea"]), 6, 6))
    r, J0, J1 = po.edges_eval(g["init"], g["ea"], g["eb"], g["rel"], S)
    for e in range(0, len(g["ea"]), 3):
        r1, a, b = po.edge_eval(g["init"][g["ea"][e]], g["init"][g["eb"][e]], g["rel"][e], S[e])
        assert np.abs(r[e] - r1).max() <= 1e-12 * max(1.0, np.abs(r1).max()) and np.abs(J0[e] - a).max() <= 1e-12 * np.abs(a).max() and np.abs(J1[e] - b).max() <= 1e-12 * np.abs(b).max()
