#!/usr/bin/env python
"""Voxel-grid SDF rows (KIN_PRIM_GRID) against the analytic fridge on the B200.

Fetch with the 16-sphere fixture, SoA, FP64 and FP32.  The fridge of data/fridge.urdf four ways:
  boxes      the 7 boxes (the reference's UnionSDF)
  grid 2cm   GridSDF.from_sdf of the boxes, 2.4 m cubed at 2 cm (121^3 samples)
  grid 1cm   the same at 1 cm (241^3 samples)
  grid+boxes the 2 cm grid and the 7 boxes in one union
Timed per scene, alternated round by round in one process, CUDA events, median of the rounds:
  coll FD / coll AN   kin_eval, collision only (values + gradients), forward-difference / analytic gradient
  fused               kin_eval FK of the gripper + its Jacobian + collision (FD), one launch
  ik                  collision-constrained inverse_kinematics_batch at 2^LOG_IK targets (FP64, 40 + 60 iterations)
  points/s            kin_sdf_points over 2^24 random points around the fridge (FP64, values + FD gradient)
Usage: python profiles/bench_grid_sdf.py [log2 N (22 23 24)...] [--rounds R] [--log-ik L]"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

import kinematics_jl_b200 as K
from kinematics_jl_b200.device import current_q, device_model, evaluate
import scene_fetch as SF

GRID_POSE = np.eye(4)
GRID_POSE[:3, 3] = [0.6, 0.0, 0.9]


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else "unknown"


def timed(fn, reps=3):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    args = sys.argv[1:]
    rounds, log_ik = 5, 20
    if "--rounds" in args:
        i = args.index("--rounds"); rounds = int(args[i + 1]); del args[i:i + 2]
    if "--log-ik" in args:
        i = args.index("--log-ik"); log_ik = int(args[i + 1]); del args[i:i + 2]
    logs = [int(a) for a in args] or [22, 23, 24]
    print("card, power limit: %s" % card())
    m, joints, sscc = SF.product_fetch(False)
    boxes = SF.product_fridge_sdf()
    g2 = K.GridSDF.from_sdf(boxes, K.Transform(GRID_POSE), (121, 121, 121), 0.02)
    g1 = K.GridSDF.from_sdf(boxes, K.Transform(GRID_POSE), (241, 241, 241), 0.01)
    scenes = {"boxes": boxes, "grid 2cm": g2, "grid 1cm": g1, "grid+boxes": K.UnionSDF([g2, boxes])}
    print("grid MB: 2cm %.1f, 1cm %.1f" % (121 ** 3 * 4 / 2 ** 20, 241 ** 3 * 4 / 2 ** 20))
    gl = K.find_link(m, "gripper_link").id
    lo, hi = SF.joint_limits(joints)
    rng = np.random.default_rng(0)
    for dt in (torch.float64, torch.float32):
        for lg in logs:
            N = 1 << lg
            q = torch.as_tensor(lo + (hi - lo) * rng.random((N, len(joints))), dtype=dt, device="cuda")
            K.set_joint_angles(m, joints, q.t().contiguous().t())          # SoA
            res = {k: {"coll FD": [], "coll AN": [], "fused": []} for k in scenes}
            for r in range(rounds + 1):
                for name, sdf in scenes.items():
                    K.compute_coll_dists(sscc, joints, sdf)                 # puts this scene's table into the model
                    dm = device_model(m)
                    Qc, ql, n = current_q(m)
                    calls = {"coll FD": dict(collision=True, grad_mode=K.GRAD_FD),
                             "coll AN": dict(collision=True, grad_mode=K.GRAD_ANALYTIC),
                             "fused": dict(collision=True, fk_links=[gl], jac_links=[gl])}
                    for key, kw in calls.items():
                        t = timed(lambda: evaluate(dm, Qc, ql, n, **kw))
                        if r > 0:                                           # round 0 warms up (JIT, L2)
                            res[name][key].append(t)
            for name in scenes:
                print("%s 2^%d %-10s " % ("FP64" if dt == torch.float64 else "FP32", lg, name) +
                      "  ".join("%s %.3f ms" % (k, np.median(v)) for k, v in res[name].items()))
            del q
            torch.cuda.empty_cache()
    # constrained IK, FP64
    link = K.find_link(m, "gripper_link")
    N = 1 << log_ik
    tg = np.zeros((N, 6))
    tg[:, 0], tg[:, 1], tg[:, 2] = rng.uniform(0.75, 1.0, N), rng.uniform(-0.15, 0.15, N), rng.uniform(1.12, 1.35, N)
    q0 = torch.as_tensor(np.tile([0.2, 0, 0, 0, 0.5, 0, 0.5, 0], (N, 1)), dtype=torch.float64, device="cuda")
    tgt = torch.as_tensor(tg, device="cuda")
    ik = {k: [] for k in scenes}
    for r in range(3):
        for name, sdf in scenes.items():
            t = timed(lambda: K.inverse_kinematics_batch(m, link, joints, tgt, q0, iters=40, sscc=sscc, sdf=sdf), reps=1)
            if r > 0:
                ik[name].append(t)
    for name in scenes:
        print("IK 2^%d %-10s %.1f ms" % (log_ik, name, np.median(ik[name])))
    # points
    P = torch.as_tensor(GRID_POSE[:3, 3] + (np.random.default_rng(1).random((1 << 24, 3)) - 0.5) * 2.4, device="cuda")
    for name, sdf in scenes.items():
        sdf.gradient(P)
        t = np.median([timed(lambda: sdf.gradient(P)) for _ in range(rounds)])
        print("points %-10s %.3f ms  %.2f Gpoints/s" % (name, t, (1 << 24) / t / 1e6))


if __name__ == "__main__":
    main()
