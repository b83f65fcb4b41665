"""A/B of the constant-row fill (kin_gen_skeleton.cuh: kin_const_fill_kernel) on the bench headline, in one process.

2^24 Fetch configurations, SoA, float64 (bench.py's inputs), FK-all + gripper Jacobian: every row stored per thread
(KIN_JIT_CONST_FILL=0) against the 175 constant rows written by the fill kernel (the default).  Each round times STEPS
kin_eval calls of each variant (CUDA events, ms per call); rounds alternate the variants; median / min / max over the
rounds.  The outputs of the two are compared bit for bit.
Usage: python profiles/ab_const_fill.py [rounds] [steps]"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import kinematics_jl_b200 as K                    # noqa: E402
from kinematics_jl_b200 import lib as L          # noqa: E402
from kinematics_jl_b200.device import device_model  # noqa: E402
import scene_fetch                               # noqa: E402

N, N_DOF, N_LINKS = 1 << 24, 8, 25


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 9
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout, flush=True)
    dev = torch.device("cuda", 0)
    m, joints, sscc = scene_fetch.product_fetch(False)
    K.set_joint_angles(m, joints, torch.zeros((1, N_DOF), dtype=torch.float64, device=dev))
    dm = device_model(m)
    lib = L.lib()
    g = torch.Generator(device=dev).manual_seed(0)
    lo_np, hi_np = scene_fetch.joint_limits(joints)
    lo, hi = torch.tensor(lo_np, device=dev), torch.tensor(hi_np, device=dev)
    Q = lo[:, None] + (hi - lo)[:, None] * torch.rand((N_DOF, N), generator=g, device=dev, dtype=torch.float64)
    T = torch.empty((N_LINKS * 12, N), dtype=torch.float64, device=dev)
    J = torch.empty((6 * N_DOF, N), dtype=torch.float64, device=dev)
    fk = np.arange(1, N_LINKS + 1, dtype=np.int32)
    jac = np.array([K.find_link(m, "gripper_link").id], dtype=np.int32)
    ip = C.POINTER(C.c_int32)
    stream = torch.cuda.current_stream(dev)
    c = L.KinCall()
    c.precision, c.layout, c.n, c.q = L.F64, L.SOA, N, Q.data_ptr()
    c.n_fk_links, c.fk_links, c.T_out = N_LINKS, fk.ctypes.data_as(ip), T.data_ptr()
    c.n_jac_links, c.jac_links, c.J_out, c.with_rot = 1, jac.ctypes.data_as(ip), J.data_ptr(), 1
    c.truncation_dist = float("inf")
    c.stream = stream.cuda_stream

    def run(fill, n_steps):
        os.environ["KIN_JIT_CONST_FILL"] = fill
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record(stream)
        for _ in range(n_steps):
            L.check(lib.kin_eval(dm.h, C.byref(c)))
        ev[1].record(stream)
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) / n_steps

    run("0", 3)                                      # compile + warm up; the outputs of both variants compared
    ref = (T.clone(), J.clone())
    T.fill_(-1.0), J.fill_(-1.0)
    run("1", 3)
    same = torch.equal(ref[0].view(torch.int64), T.view(torch.int64)) and torch.equal(ref[1].view(torch.int64), J.view(torch.int64))
    print("outputs bitwise equal, fill off / on:", same, flush=True)
    del ref
    ms = {"0": [], "1": []}
    for _ in range(rounds):
        for f in ms:
            ms[f].append(run(f, steps))
    print("%-10s %9s %9s %9s   (%d rounds x %d calls, 2^24 configurations, alternating)" % ("fill", "med ms", "min ms", "max ms", rounds, steps))
    for f, x in ms.items():
        x = sorted(x)
        print("%-10s %9.4f %9.4f %9.4f" % ({"0": "off", "1": "on"}[f], x[len(x) // 2], x[0], x[-1]))
    pa, pb = np.median(ms["0"]), np.median(ms["1"])
    spread = max(max(x) - min(x) for x in ms.values())
    print("on / off = %.4f  (gain %.3f ms, largest min-max spread %.3f ms)" % (pb / pa, pa - pb, spread))


if __name__ == "__main__":
    main()
