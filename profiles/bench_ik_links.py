#!/usr/bin/env python
"""kin_ik_solve_links (batched IK with several target links per problem) on the B200.

Dual-arm model, fixed base (15 columns) and planar base (18 columns), 2^18 problems: both tool targets (l_tool and
r_tool, with rotation) are the poses of ONE random in-limit configuration whose pairs are all >= 0.05 apart, so the pair
is jointly reachable; seeds are random in-limit configurations.  Solves, alternated in one process, CUDA events, median
of the timed rounds:
  (a)  l_tool only            kin_ik_solve (generated one-launch kernel), the right tool is a passenger
  (b)  both tools, pose only  kin_ik_solve_links, generated one-launch kernel (staged)
  (b') both tools, pose only  the same through the (kin_eval, step kernel) loop (KIN_DISABLE_JIT), for the path selection
  (c)  both + self            kin_ik_solve_links, self_collision = 1 (145 pairs)
  (d)  both + boxes + self    kin_ik_solve_links, self_collision = 1, collision = 1 (the model's three boxes)
(a), (b), (b') run 40 iterations at most, (c) and (d) 60, all from the seeds.
Reported per solve: ms, the share reaching both targets (every residual of both tools <= 1e-3; for (a) the left tool's
share is given as well), the share clear (every pair >= margin - 1e-3, with (d) every sphere too), mean iterations and,
for the loop, the mean active-list length per iteration derived from the returned iterations (bench_ik_self.py).
Usage: python profiles/bench_ik_links.py [log2 N (18)] [rounds (5)]"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, HERE)
import numpy as np
import torch

import kinematics_jl_b200 as K
import scene_fetch as SF
from bench_ik_self import mean_active, random_q

MARGIN, ITERS, COLL_ITERS, FTOL = 0.02, 40, 60, 1e-10


def rpy_targets(T):
    Rm, p = T[:, :, :3], T[:, :, 3]
    yaw = torch.atan2(Rm[:, 1, 0], Rm[:, 0, 0])
    pitch = torch.atan2(-Rm[:, 2, 0], torch.sqrt(Rm[:, 2, 1] ** 2 + Rm[:, 2, 2] ** 2))
    s, c = torch.sin(yaw), torch.cos(yaw)
    roll = torch.atan2(Rm[:, 0, 2] * s - Rm[:, 1, 2] * c, Rm[:, 1, 1] * c - Rm[:, 0, 1] * s)
    return torch.cat([p, roll[:, None], pitch[:, None], yaw[:, None]], dim=1)


def problems(m, joints, sscc, links, N, pairs, seed):
    q, n = [], 0
    while n < N:
        qc = random_q(m, joints, 2 * N, seed)
        seed += 1
        K.set_joint_angles(m, joints, qc)
        d, _ = K.compute_self_coll_summary(sscc, joints, pairs)
        q.append(qc[d >= 0.05])
        n += q[-1].shape[0]
    qt = torch.cat(q)[:N].contiguous()
    K.set_joint_angles(m, joints, qt)
    tg = torch.cat([rpy_targets(K.get_transform(m, l)) for l in links], dim=1).contiguous()
    return tg, random_q(m, joints, N, seed + 1000).contiguous()


def max_err(m, joints, link, q, tg):
    K.set_joint_angles(m, joints, q)
    v, _ = K.pose_constraint(m, link, joints, tg, True)
    v[:, 3:] = torch.remainder(v[:, 3:] + np.pi, 2 * np.pi) - np.pi
    return v.abs().amax(dim=1)


def loop(fn):
    os.environ["KIN_DISABLE_JIT"] = "1"
    try:
        return fn()
    finally:
        del os.environ["KIN_DISABLE_JIT"]


def run(name, m, joints, sscc, sdf, N, pairs, rounds):
    links = [K.find_link(m, "l_tool"), K.find_link(m, "r_tool")]
    tg, q0 = problems(m, joints, sscc, links, N, pairs, 1)
    tg_l = tg[:, :6].contiguous()
    K.compute_coll_dists(sscc, joints, sdf)                      # spheres + boxes on the device model
    solves = {
        "(a)  l_tool only": lambda: K.ik_solve_device(m, links[0], joints, tg_l, q0, iters=ITERS, ftol=FTOL),
        "(b)  both, generated": lambda: K.ik_solve_device(m, links, joints, tg, q0, iters=ITERS, ftol=FTOL),
        "(b') both, loop": lambda: loop(lambda: K.ik_solve_device(m, links, joints, tg, q0, iters=ITERS, ftol=FTOL)),
        "(c)  both + self": lambda: K.ik_solve_device(m, links, joints, tg, q0, iters=COLL_ITERS, ftol=FTOL, sscc=sscc,
                                                      self_margin=MARGIN, self_pairs=pairs),
        "(d)  both + boxes + self": lambda: K.ik_solve_device(m, links, joints, tg, q0, iters=COLL_ITERS, ftol=FTOL, sscc=sscc,
                                                              sdf=sdf, margin=MARGIN, self_margin=MARGIN, self_pairs=pairs),
    }
    times, outs = {k: [] for k in solves}, {}
    for r in range(rounds + 1):                                  # round 0: warm-up (module loads, JIT, pool growth)
        for k, f in solves.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            outs[k] = f()
            b.record()
            torch.cuda.synchronize()
            if r > 0:
                times[k].append(a.elapsed_time(b))
    print("\n%s: N = %d problems, %d columns, %d pairs, %d spheres, %d boxes; median of %d rounds after 1 warm-up round"
          % (name, N, q0.shape[1], len(pairs), len(sscc.sphere_links), len(sdf.world_primitives()[0]), rounds))
    for k, out in outs.items():
        q, f, its = out[0], out[1], out[2]
        el = max_err(m, joints, links[0], q, tg[:, :6])
        er = max_err(m, joints, links[1], q, tg[:, 6:])
        both = (el < 1e-3) & (er < 1e-3)
        K.set_joint_angles(m, joints, q)
        sd, _ = K.compute_self_coll_summary(sscc, joints, pairs)
        clear = sd >= MARGIN - 1e-3
        if k.startswith("(d)"):
            clear = clear & (out[3] >= MARGIN - 1e-3)
        line = "  %-26s %9.2f ms  both reached %5.1f %%  clear %5.1f %%  both + clear %5.1f %%  mean its %5.1f" % (
            k, float(np.median(times[k])), 100 * both.double().mean(), 100 * clear.double().mean(),
            100 * (both & clear).double().mean(), float(its.double().mean()))
        if k.startswith("(a)"):
            line += "  (l_tool reached %5.1f %%)" % (100 * (el < 1e-3).double().mean())
        if k[1] in "cd" or k.startswith("(b')"):
            n_it = COLL_ITERS if k[1] in "cd" else ITERS
            stopped = (f < FTOL).cpu().numpy()
            if k[1] in "cd":
                stopped = stopped & clear.cpu().numpy()
            ma = mean_active(its.cpu().numpy(), stopped, n_it)
            line += "  mean active list %8.0f (%4.1f %% of N)" % (ma, 100 * ma / N)
        print(line)
    del outs
    torch.cuda.empty_cache()


def main():
    la = int(sys.argv[1]) if len(sys.argv) > 1 else 18
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    print(smi.stdout.strip())
    for with_base in (False, True):
        m, joints, sscc, sdf = SF.product_dual_arm(with_base)
        run("dual arm, %s base" % ("planar" if with_base else "fixed"), m, joints, sscc, sdf, 1 << la,
            K.self_collision_pairs(sscc, joints), rounds)


if __name__ == "__main__":
    main()
