#!/usr/bin/env python
"""kin_self_collision (self-collision between the collision spheres, an extension) on the B200, SoA, FP64 and FP32, on
the dual-arm model (15 columns, default pairs: 145) and on Fetch with the 8 arm joints (80 pairs), three variants:
  (a) dmin / amin only  -- the collision-check workload: 12 (FP64) or 8 (FP32) bytes written per configuration
  (b) vals              -- P values per configuration
  (c) vals + grads      -- P (1 + n_dof) values per configuration
alternated in the same process with kin_collision (values + gradients against the model's boxes, clean scratch) and
kin_collision_summary on the same batch, so that the new call sits next to a known number.  CUDA events, two warm-up
rounds, median of the timed rounds.  Bytes per configuration are counted from the shapes (q read + outputs written);
(b) / (c) are compared with the 7.7 TB/s HBM3e data-sheet bandwidth, (a) is reported as pairs per second.
Usage: python profiles/bench_self_collision.py [log2 N (default 20)] [rounds (default 7)]"""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import device_model
import scene_fetch as SF

HBM = 7.7e12


def configs(joints, N, seed):
    lo, hi = SF.joint_limits(joints)
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = torch.rand((len(joints), N), dtype=torch.float64, device="cuda", generator=g)     # SoA storage (n_dof, N)
    return torch.as_tensor(lo, device="cuda")[:, None] + torch.as_tensor(hi - lo, device="cuda")[:, None] * u


def model(name):
    if name == "dual_arm":
        m, joints, sscc, sdf = SF.product_dual_arm(False)
    else:
        m, joints, sscc = SF.product_fetch(False)
        sdf = SF.product_fridge_sdf()
    K.set_joint_angles(m, joints, np.zeros(len(joints)))
    K.compute_coll_dists(sscc, joints, sdf)                  # spheres + boxes on the device model
    K.compute_self_coll_dists(sscc, joints)                  # default pair table
    return m, joints, sscc, device_model(m)


def main():
    logn = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    N = 1 << logn
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    print(smi.stdout.strip())
    lib = L.lib()
    st = torch.cuda.current_stream().cuda_stream
    print("N = %d configurations per call, SoA, median of %d alternated rounds after 2 warm-up rounds" % (N, rounds))
    for name in ("dual_arm", "fetch"):
        m, joints, sscc, dm = model(name)
        P, S, nd = dm.n_self_pairs, dm.n_spheres, dm.n_dof
        for dt, prec in ((torch.float64, L.F64), (torch.float32, L.F32)):
            es = 8 if dt == torch.float64 else 4
            Q = configs(joints, N, 1).to(dt).contiguous()        # (nd, N): SoA, ld = N
            V = torch.empty((P, N), dtype=dt, device="cuda")
            G = torch.empty((P, nd, N), dtype=dt, device="cuda")
            dmin = torch.empty(N, dtype=dt, device="cuda")
            amin = torch.empty(N, dtype=torch.int32, device="cuda")
            EV = torch.empty((S, N), dtype=dt, device="cuda")
            EG = torch.empty((S, nd, N), dtype=dt, device="cuda")
            inf = float("inf")
            calls = {
                "self (a) dmin/amin": (lambda: lib.kin_self_collision(dm.h, prec, L.SOA, Q.data_ptr(), N, inf, 0.0, None, None,
                                                                       dmin.data_ptr(), amin.data_ptr(), st), es + 4),
                "self (b) vals": (lambda: lib.kin_self_collision(dm.h, prec, L.SOA, Q.data_ptr(), N, inf, 0.0, V.data_ptr(), None,
                                                                  None, None, st), P * es),
                "self (c) vals+grads": (lambda: lib.kin_self_collision(dm.h, prec, L.SOA, Q.data_ptr(), N, inf, 0.0, V.data_ptr(),
                                                                        G.data_ptr(), None, None, st), P * (1 + nd) * es),
                # lib.py declares no argtypes for kin_collision: the arguments carry their C types here
                "kin_collision vals+grads": (lambda: lib.kin_collision(dm.h, C.c_int32(prec), C.c_int32(L.SOA), C.c_void_p(Q.data_ptr()),
                                                                       C.c_int64(N), C.c_double(inf), C.c_int32(L.GRAD_FD),
                                                                       C.c_int32(L.SCRATCH_CLEAN), C.c_void_p(EV.data_ptr()),
                                                                       C.c_void_p(EG.data_ptr()), None, C.c_void_p(st)),
                                             S * (1 + nd) * es),
                "kin_collision_summary": (lambda: lib.kin_collision_summary(dm.h, prec, L.SOA, Q.data_ptr(), N, 0.0, dmin.data_ptr(),
                                                                            amin.data_ptr(), None, st), es + 4),
            }
            times = {k: [] for k in calls}
            for r in range(rounds + 2):
                for k, (f, _) in calls.items():
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    L.check(f())
                    b.record()
                    torch.cuda.synchronize()
                    if r >= 2:
                        times[k].append(a.elapsed_time(b))
            print("\n%s, %s: P = %d pairs, S = %d spheres, n_dof = %d" % (name, "FP64" if es == 8 else "FP32", P, S, nd))
            for k, (_, out_bytes) in calls.items():
                ms = float(np.median(times[k]))
                byts = nd * es + out_bytes
                line = "  %-26s %8.3f ms  %6.1f ns/config  %7d B/config  %6.2f TB/s (%4.1f %% of 7.7)" % (
                    k, ms, ms * 1e6 / N, byts, byts * N / (ms * 1e-3) / 1e12, 100 * byts * N / (ms * 1e-3) / HBM)
                if k.startswith("self (a)"):
                    line += "  %.3g pairs/s" % (P * N / (ms * 1e-3))
                print(line)
            del V, G, EV, EG
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
