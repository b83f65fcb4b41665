#!/usr/bin/env python
"""kin_ik_solve_self (batched IK with the self-collision pairs as a hard constraint) on the B200.

Dual-arm model (l_tool targets, default 145-pair table), fixed base (15 columns) and planar base (18 columns), 2^18
problems: targets are the tool poses of random in-limit configurations whose pairs are all >= 0.05 apart, seeds are
random in-limit configurations.  Three solves, alternated in one process, CUDA events, median of the timed rounds:
  (a) pose only           kin_ik_solve, collision = 0 (the generated one-launch kernel)
  (b) pose + self         kin_ik_solve_self, collision = 0
  (c) pose + boxes + self kin_ik_solve_self, collision = 1 (the model's three boxes)
(b) and (c) start from the seeds, like (a), with 60 iterations at most; (a) runs 40.  Then Fetch (gripper_link, 8 arm
joints) at 2^20 with the 64-pair table (the default policy minus the elbow / wrist pair that overlaps in every
configuration) and the fridge, (a) / (b) / (c) likewise.
Reported per solve: ms, the share of problems reached (f <= 1e-6, i.e. every residual <= 1e-3), the share clear (every
pair, and with (c) every sphere, >= margin - 1e-3), and the mean active-list length per iteration, derived from the
returned iterations: a problem that stopped at iteration k leaves the list at the first compaction after k (1, 2, 3, 4,
6, 8, 12, ...); one that did not stop stays to the end.
Usage: python profiles/bench_ik_self.py [log2 N dual arm (18)] [log2 N Fetch (20)] [rounds (5)]"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

import kinematics_jl_b200 as K
import scene_fetch as SF

MARGIN, ITERS, COLL_ITERS, FTOL = 0.02, 40, 60, 1e-10


def compactions(iters):
    """Iterations at which the active list is rebuilt (kin_b200.cu: ik_solve_coll)."""
    out, it, step = [], 1, 1
    while it <= iters:
        out.append(it)
        if it >= 4 and (it & (it - 1)) == 0:
            step = it // 2
        it += step
    return np.array(out)


def mean_active(its, stopped, iters):
    """Mean over iterations 0..iters of the active-list length implied by the stop iterations."""
    c = compactions(iters)
    leave = np.full(its.shape, iters + 1)
    k = np.searchsorted(c, its[stopped], side="right")          # first compaction after the stop iteration
    leave[stopped] = np.where(k < len(c), c[np.minimum(k, len(c) - 1)], iters + 1)
    return float(np.minimum(leave, iters + 1).sum()) / (iters + 1)


def random_q(m, joints, N, seed):
    lo, hi = SF.joint_limits(joints)
    if m.with_base:                                              # planar base x, y, theta (inverse_kinematics._seed_limits)
        lo, hi = np.concatenate([lo, [-1.0, -1.0, -np.pi]]), np.concatenate([hi, [1.0, 1.0, np.pi]])
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = torch.rand((N, len(lo)), dtype=torch.float64, device="cuda", generator=g)
    return torch.as_tensor(lo, device="cuda") + torch.as_tensor(hi - lo, device="cuda") * u


def problems(m, joints, sscc, link, N, pairs, seed):
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
    T = K.get_transform(m, link)                                 # (N, 3, 4)
    Rm, p = T[:, :, :3], T[:, :, 3]
    yaw = torch.atan2(Rm[:, 1, 0], Rm[:, 0, 0])
    pitch = torch.atan2(-Rm[:, 2, 0], torch.sqrt(Rm[:, 2, 1] ** 2 + Rm[:, 2, 2] ** 2))
    s, c = torch.sin(yaw), torch.cos(yaw)
    roll = torch.atan2(Rm[:, 0, 2] * s - Rm[:, 1, 2] * c, Rm[:, 1, 1] * c - Rm[:, 0, 1] * s)
    tg = torch.cat([p, roll[:, None], pitch[:, None], yaw[:, None]], dim=1).contiguous()
    return tg, random_q(m, joints, N, seed + 1000).contiguous()


def run(name, m, joints, sscc, sdf, link, N, pairs, rounds):
    tg, q0 = problems(m, joints, sscc, link, N, pairs, 1)
    K.compute_coll_dists(sscc, joints, sdf)                      # spheres + boxes on the device model
    solves = {
        "(a) pose only": lambda: K.ik_solve_device(m, link, joints, tg, q0, iters=ITERS, ftol=FTOL),
        "(b) pose + self": lambda: K.ik_solve_device(m, link, joints, tg, q0, iters=COLL_ITERS, ftol=FTOL, sscc=sscc,
                                                     self_margin=MARGIN, self_pairs=pairs),
        "(c) pose + boxes + self": lambda: K.ik_solve_device(m, link, joints, tg, q0, iters=COLL_ITERS, ftol=FTOL, sscc=sscc,
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
        reached = f <= 1e-6
        K.set_joint_angles(m, joints, q)
        sd, _ = K.compute_self_coll_summary(sscc, joints, pairs)
        clear = sd >= MARGIN - 1e-3
        if k.startswith("(c)"):
            clear = clear & (out[3] >= MARGIN - 1e-3)
        line = "  %-24s %9.2f ms  reached %5.1f %%  clear %5.1f %%  both %5.1f %%  mean its %5.1f" % (
            k, float(np.median(times[k])), 100 * reached.double().mean(), 100 * clear.double().mean(),
            100 * (reached & clear).double().mean(), float(its.double().mean()))
        if not k.startswith("(a)"):
            stopped = (reached & clear).cpu().numpy()           # f < ftol and every constraint within ctol implies both
            line += "  mean active list %8.0f (%4.1f %% of N)" % (mean_active(its.cpu().numpy(), stopped, COLL_ITERS),
                                                                  100 * mean_active(its.cpu().numpy(), stopped, COLL_ITERS) / N)
        print(line)
    del outs
    torch.cuda.empty_cache()


def main():
    la = int(sys.argv[1]) if len(sys.argv) > 1 else 18
    lf = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    print(smi.stdout.strip())
    for with_base in (False, True):
        m, joints, sscc, sdf = SF.product_dual_arm(with_base)
        run("dual arm, %s base" % ("planar" if with_base else "fixed"), m, joints, sscc, sdf, K.find_link(m, "l_tool"), 1 << la,
            K.self_collision_pairs(sscc, joints), rounds)
    m, joints, sscc = SF.product_fetch(False)
    run("Fetch + fridge", m, joints, sscc, SF.product_fridge_sdf(), K.find_link(m, "gripper_link"), 1 << lf,
        K.self_collision_pairs(sscc, joints, ignore=[("wrist_flex_link", "elbow_flex_link")]), rounds)


if __name__ == "__main__":
    main()
