"""Freezes outputs of the REFERENCE's own code (oracle/_ref/libd2ref.so, built from the reference sources by
oracle/Makefile.ref) on the seeded cases of tests/test_ref_pin.py into tests/golden/ref_factors.npz, and on those of the
remaining reference comparisons (preintegration, manifold helpers, the device-vs-reference windows, the pose-graph functor and
g2o reader / writer) into tests/golden/ref_extra.npz.  The tests compare with these where the library is absent.
Run where the reference sources are available:  python tests/golden/make_ref_golden.py"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import test_gpu_vs_reference as tg  # noqa: E402
import test_pgo as tp  # noqa: E402
import test_ref_pin as t  # noqa: E402
from oracle import ref  # noqa: E402

out = {}
for i, c in enumerate(t.proj_cases()):
    r, Js, tb = ref.proj_eval(c["typ"], c["pts_i"], c["pts_j"], c["vel_i"], c["vel_j"], c["td_i"], c["td_j"], c["depth"], t.ref_params(c))
    out[f"proj{i}_r"] = r; out[f"proj{i}_tb"] = tb
    for k, J in enumerate(Js):
        out[f"proj{i}_J{k}"] = J
for i, c in enumerate(t.imu_cases()):
    pre = ref.preintegrate(c["dt"], c["acc"], c["gyr"], c["ba0"], c["bg0"])
    r, Js, si = ref.imu_eval(pre, c["ba0"], c["bg0"], c["pi"], c["sbi"], c["pj"], c["sbj"])
    out[f"imu{i}_pre_jacobian"] = pre["jacobian"]; out[f"imu{i}_pre_covariance"] = pre["covariance"]
    out[f"imu{i}_sqrt_info"] = si; out[f"imu{i}_r"] = r
    for k, J in enumerate(Js):
        out[f"imu{i}_J{k}"] = J
for i, c in enumerate(t.cons_cases()):
    r, J = ref.consensus_eval(c["z"][:3], c["z"][3:7], c["tt"], c["th"], c["rho_T"], c["rho_theta"], c["x"])
    out[f"cons{i}_r"] = r; out[f"cons{i}_J"] = J
for i, c in enumerate(t.relpose_cases()):
    r, Ja, Jb = ref.relpose_ad_eval(c["pa"], c["pb"], c["rel"], c["S"])
    out[f"relpose{i}_r"] = r; out[f"relpose{i}_Ja"] = Ja; out[f"relpose{i}_Jb"] = Jb
for i, c in enumerate(t.loss_cases()):
    r, J = ref.loss_correct(c["r"], c["J"], c["a"])
    out[f"loss{i}_r"] = r; out[f"loss{i}_J"] = J
for i, c in enumerate(t.prior_cases()):
    out[f"prior{i}_r"], out[f"prior{i}_J"] = ref.prior_eval(c["kinds"], c["x0"], c["x"], c["A"], c["b"])
for i, c in enumerate(t.relpose4d_cases()):
    out[f"relpose4d{i}_r"], out[f"relpose4d{i}_Ja"], out[f"relpose4d{i}_Jb"] = ref.relpose4d_eval(c["pa"], c["pb"], c["rel"], c["S"])
ref.configure()
for i, kw in enumerate(t.MARG_CASES):
    pr = t.synth.make_window(**kw)
    out[f"marg{i}_refs"], out[f"marg{i}_x0"], out[f"marg{i}_J"], out[f"marg{i}_e0"] = ref.marginalize(pr, [int(pr["frame_ids"][0])])
_, present, traj = t.admm_trajectory()
out["admm_z"], out["admm_tilde"], out["admm_res"] = ref.admm_replay(present, traj, t.ADMM_KW["relaxation_alpha"], t.ADMM_KW["rho_frame_T"], t.ADMM_KW["rho_frame_theta"])
np.savez_compressed(os.path.join(HERE, "ref_factors.npz"), **out)
print("wrote", len(out), "arrays")

extra = {}
for i, c in enumerate(t.imu_cases()):
    pre = ref.preintegrate(c["dt"], c["acc"], c["gyr"], c["ba0"], c["bg0"])
    for k in ("sum_dt", "delta_p", "delta_q", "delta_v"):
        extra[f"imu{i}_pre_{k}"] = pre[k]
extra["manifold_plus"], extra["manifold_plus_jacobian"], extra["manifold_average_quat"] = t.reference_manifold(*t.manifold_cases())
for c, case in enumerate(tg.PROJ_CASES):
    pr = t.synth.make_window(**case)
    idx = tg.proj_sample(pr)
    extra[f"dev_proj{c}_idx"] = idx
    extra[f"dev_proj{c}_r"], extra[f"dev_proj{c}_J"] = tg.reference_proj(pr, idx)
extra["dev_imu_r"], extra["dev_imu_J"], extra["dev_imu_sqrt_info"] = tg.reference_imu(t.synth.make_window(**tg.IMU_CASE))
extra["functor_r"], extra["functor_Ja"], extra["functor_Jb"] = tp.reference_functor(*tp.functor_case())
with tempfile.TemporaryDirectory() as d:
    _, _, agents = tp.g2o_agents_case(d)
    extra.update({f"g2o_agents_{k}": v for k, v in tp.reference_g2o_reads(d, agents).items()})
    path = os.path.join(d, "out.g2o")
    tp.reference_g2o_write(path, *tp.reference_written_case())
    with open(path, "rb") as f:
        extra["g2o_written_file"] = np.frombuffer(f.read(), np.uint8)
np.savez_compressed(os.path.join(HERE, "ref_extra.npz"), **extra)
print("wrote", len(extra), "arrays")
