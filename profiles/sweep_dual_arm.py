"""A dual-arm mechanism (data/dual_arm.urdf: 15 columns, 18 with the planar base, 19 spheres, 3 boxes): the fused
call and the collision-only call, interpreting kernel against the specialised one, SoA.
python profiles/sweep_dual_arm.py [log2 n]
SWEEP_JIT_ONLY=1 with KIN_JIT_BLOCK / KIN_JIT_MINB: launch-shape variants of the specialised kernel."""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import kinematics_jl_b200 as K  # noqa: E402
import scene_fetch  # noqa: E402
from kinematics_jl_b200 import lib as L  # noqa: E402
from kinematics_jl_b200.device import device_model  # noqa: E402

N = 1 << (int(sys.argv[1]) if len(sys.argv) > 1 else 21)
F32 = bool(os.environ.get("SWEEP_F32"))
DT, RS = (torch.float32, 4) if F32 else (torch.float64, 8)
dev = torch.device("cuda", 0)
lib = L.lib()
stream = torch.cuda.current_stream(dev)
ip = C.POINTER(C.c_int32)
for with_base in (False, True):
    m, joints, sscc, sdf = scene_fetch.product_dual_arm(with_base)
    nd, S, nl = len(joints) + (3 if with_base else 0), len(sscc.sphere_radii), len(m.links)
    K.set_joint_angles(m, joints, torch.zeros((1, nd), dtype=torch.float64, device=dev))
    K.compute_coll_dists(sscc, joints, sdf)
    dm = device_model(m)
    g = torch.Generator(device=dev).manual_seed(0)
    Q = (2.0 * torch.rand((nd, N), generator=g, device=dev, dtype=torch.float64) - 1.0).to(DT)
    T = torch.empty((12 * nl, N), dtype=DT, device=dev)
    V = torch.empty((S, N), dtype=DT, device=dev)
    G = torch.empty((S * nd, N), dtype=DT, device=dev)
    fk = np.array([l.id for l in m.links], dtype=np.int32)
    for fused in (False, True):
        res = {}
        for jit in ((True,) if os.environ.get("SWEEP_JIT_ONLY") else (False, True)):
            os.environ.pop("KIN_DISABLE_JIT", None)
            os.environ.pop("KIN_FORCE_JIT", None)
            os.environ["KIN_FORCE_JIT" if jit else "KIN_DISABLE_JIT"] = "1"
            c = L.KinCall()
            c.precision, c.layout, c.n, c.q = (L.F32 if F32 else L.F64), L.SOA, N, Q.data_ptr()
            if fused:
                c.n_fk_links, c.fk_links, c.T_out = nl, fk.ctypes.data_as(ip), T.data_ptr()
            c.truncation_dist = float("inf")
            c.vals_out, c.grads_out = V.data_ptr(), G.data_ptr()
            c.stream = stream.cuda_stream
            for _ in range(3):
                L.check(lib.kin_eval(dm.h, C.byref(c)))
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(10):
                L.check(lib.kin_eval(dm.h, C.byref(c)))
            b.record(stream)
            torch.cuda.synchronize()
            regs, smem, block, grid = (C.c_int32() for _ in range(4))
            L.check(lib.kin_query_launch(dm.h, C.byref(c), C.byref(regs), C.byref(smem), C.byref(block), C.byref(grid)))
            ms = a.elapsed_time(b) / 10
            byts = RS * (nd + S + S * nd + (12 * nl if fused else 0))
            res[jit] = (V.clone(), G.clone())
            print("%s base=%d %s %s: %.3f ms per 2^%d (%.3e configs/s, %.0f GB/s algorithmic, %d B/config) block %d grid %d regs %d smem %d" %
                  ("f32" if F32 else "f64", with_base, "fused(FK all %d links + collision)" % nl if fused else "collision-only", "specialised" if jit else "interpreting",
                   ms, int(np.log2(N)), N / ms * 1e3, byts * N / ms / 1e6, byts, block.value, grid.value, regs.value, smem.value), flush=True)
        if len(res) == 2:
            print("   bitwise equal: vals %s grads %s" % (torch.equal(res[0][0], res[1][0]), torch.equal(res[0][1], res[1][1])), flush=True)
