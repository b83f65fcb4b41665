"""A/B of the FK / Jacobian schedule (kin_gen_skeleton.cuh, KSCHED: claimed tiles, inputs prefetched into L2 one epoch at
a time) against the parent commit's library (static tiles, input batches behind a grid-wide barrier), in one process.

Both libraries are loaded side by side (ctypes, one model handle each) and called on the same inputs and output buffers.
Rows: the bench headline (FK of all 25 Fetch links + gripper Jacobian, SoA, float64, 2^24 configurations); FK of the
gripper + its Jacobian (2^24; the same static schedule in both, a control); the headline call in the tiled32 layout
(2^24) and in the AoS layout (2^22).  Per row the outputs of the two libraries are compared bit for bit, then each round
times STEPS kin_eval calls of each library (CUDA events, ms per call), rounds alternating; median / min / max over the
rounds.  `--sweep` instead times the headline under the schedule knobs (KIN_JIT_EPOCH_MB, KIN_JIT_PF_DIST),
each against the parent in the same rounds; `--sizes` times the headline at 2^15 .. 2^23 with the schedule forced on
(KIN_JIT_SCHED_MIN_N=0), by the default rule, and in the parent.
Usage: python profiles/ab_sched.py PARENT_LIB [--sweep | --sizes] [rounds] [steps]
PARENT_LIB: libkin_b200.so built from the parent commit (a checkout of it, `__graft_entry__.build()` there)."""
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
from kinematics_jl_b200.device import DeviceModel  # noqa: E402
import scene_fetch                               # noqa: E402

N_DOF, N_LINKS = 8, 25
KNOBS = ("KIN_JIT_EPOCH_MB", "KIN_JIT_PF_DIST", "KIN_JIT_SCHED_MIN_N")


def load_libs(parent_path, m):
    """(library, model handle) of this tree and of the parent build; the models stay alive until the process exits."""
    new = L.lib()
    dm_new = DeviceModel(m, tuple(m._ctrl))
    so_path, allow = L.so_path, os.environ.get("KIN_ALLOW_STALE_SO")
    L._LIB, L.so_path = None, (lambda debug=False: os.path.abspath(parent_path))
    os.environ["KIN_ALLOW_STALE_SO"] = "1"      # the parent's build id is that of the parent's sources
    try:
        old = L.lib()
        dm_old = DeviceModel(m, tuple(m._ctrl))
    finally:
        L._LIB, L.so_path = new, so_path
        if allow is None:
            del os.environ["KIN_ALLOW_STALE_SO"]
    load_libs.keep = (dm_new, dm_old)           # never destroyed through the wrong library
    return {"parent": (old, dm_old.h), "this": (new, dm_new.h)}


def call(layout, n, q, T, J, fk, jac, stream, ld=0):
    ip = C.POINTER(C.c_int32)
    c = L.KinCall()
    c.precision, c.layout, c.n, c.q, c.batch_stride = L.F64, layout, n, q.data_ptr(), ld
    c.n_fk_links, c.fk_links, c.T_out = len(fk), fk.ctypes.data_as(ip), T.data_ptr()
    c.n_jac_links, c.jac_links, c.J_out, c.with_rot = 1, jac.ctypes.data_as(ip), J.data_ptr(), 1
    c.truncation_dist = float("inf")
    c.stream = stream.cuda_stream
    call.keep = (fk, jac)
    return c


def timed(lib_h, c, n_steps, stream, env=None):
    lib, h = lib_h
    for k in KNOBS:
        os.environ.pop(k, None)
    os.environ.update(env or {})
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record(stream)
    for _ in range(n_steps):
        if lib.kin_eval(h, C.byref(c)) != 0:
            raise RuntimeError(lib.kin_last_error().decode())
    ev[1].record(stream)
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / n_steps


def alternate(variants, c, rounds, steps, stream):
    """variants: {name: (lib_h, env)}; returns {name: sorted ms per call}."""
    for lh, env in variants.values():
        timed(lh, c, 3, stream, env)             # compile + warm up
    ms = {k: [] for k in variants}
    for _ in range(rounds):
        for k, (lh, env) in variants.items():
            ms[k].append(timed(lh, c, steps, stream, env))
    return {k: sorted(v) for k, v in ms.items()}


def report(title, ms, ref="parent"):
    print("%s" % title)
    for k, x in ms.items():
        print("  %-34s %9.4f %9.4f %9.4f   %s" % (k, x[len(x) // 2], x[0], x[-1],
                                                  "" if k == ref else "%.4f of %s" % (x[len(x) // 2] / ms[ref][len(ms[ref]) // 2], ref)))
    spread = max(x[-1] - x[0] for x in ms.values())
    print("  largest min-max spread %.4f ms" % spread, flush=True)


def main():
    args = sys.argv[1:]
    parent = args.pop(0)
    mode = args.pop(0) if args and args[0].startswith("--") else ""
    rounds = int(args[0]) if args else 9
    steps = int(args[1]) if len(args) > 1 else 10
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout, flush=True)
    dev = torch.device("cuda", 0)
    m, joints, _ = scene_fetch.product_fetch(False)
    K.set_joint_angles(m, joints, torch.zeros((1, N_DOF), dtype=torch.float64, device=dev))
    libs = load_libs(parent, m)
    stream = torch.cuda.current_stream(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    lo_np, hi_np = scene_fetch.joint_limits(joints)
    lo, hi = torch.tensor(lo_np, device=dev), torch.tensor(hi_np, device=dev)
    NMAX = 1 << 24
    Q = lo[:, None] + (hi - lo)[:, None] * torch.rand((N_DOF, NMAX), generator=g, device=dev, dtype=torch.float64)
    out = torch.empty(NMAX * (12 * N_LINKS + 6 * N_DOF), dtype=torch.float64, device=dev)
    fk_all = np.arange(1, N_LINKS + 1, dtype=np.int32)
    grip = K.find_link(m, "gripper_link").id
    jac = np.array([grip], dtype=np.int32)
    print("ms per call; %d rounds x %d calls, the two libraries alternating" % (rounds, steps), flush=True)

    def soa(n, fk, ld=0):
        w = ld or n
        T = out[:12 * len(fk) * w].view(12 * len(fk), w)
        J = out[12 * len(fk) * w:(12 * len(fk) + 6 * N_DOF) * w].view(6 * N_DOF, w)
        q = Q if ld == NMAX else Q[:, :n].contiguous()
        return call(L.SOA, n, q, T, J, fk, jac, stream, ld), (T, J), q

    if mode == "--sweep":
        c, _, _ = soa(NMAX, fk_all)
        variants = {"parent": (libs["parent"], None)}
        for mb in (4, 8, 16):
            for d in (0, 1, 2):
                if d == 0 and mb != 8:
                    continue                                # no prefetch: the epoch size does not matter
                variants["E %2d MB, D %d" % (mb, d)] = (libs["this"], {"KIN_JIT_EPOCH_MB": str(mb), "KIN_JIT_PF_DIST": str(d)})
        report("headline 2^24 under the schedule knobs", alternate(variants, c, rounds, steps, stream))
        return
    if mode == "--sizes":
        for lg in range(15, 24):
            c, _, _ = soa(1 << lg, fk_all, NMAX)
            variants = {"parent": (libs["parent"], None), "this, default rule": (libs["this"], None),
                        "this, claimed tiles forced": (libs["this"], {"KIN_JIT_SCHED_MIN_N": "0"})}
            report("headline 2^%d (batch_stride 2^24)" % lg, alternate(variants, c, rounds, steps, stream))
        return

    qt = Q.view(N_DOF, NMAX // 32, 32).permute(1, 0, 2).contiguous()             # tiled32: [n / 32][dof][32]
    qa = Q[:, :1 << 22].t().contiguous()                                         # AoS: [n][dof]
    rows = [("headline: FK-all + gripper J, SoA, 2^24", lambda: soa(NMAX, fk_all)),
            ("FK-gripper + J, SoA, 2^24", lambda: soa(NMAX, np.array([grip], dtype=np.int32))),
            ("FK-all + gripper J, tiled32, 2^24",
             lambda: (lambda T, J: (call(L.TILED32, NMAX, qt, T, J, fk_all, jac, stream), (T, J), qt))(
                 out[:NMAX * 300], out[NMAX * 300:NMAX * 348])),
            ("FK-all + gripper J, AoS, 2^22",
             lambda: (lambda T, J: (call(L.AOS, 1 << 22, qa, T, J, fk_all, jac, stream), (T, J), qa))(
                 out[:(1 << 22) * 300], out[(1 << 22) * 300:(1 << 22) * 348]))]
    for title, mk in rows:
        c, (T, J), q = mk()
        timed(libs["parent"], c, 1, stream)
        ref = (T.clone(), J.clone())
        T.fill_(-1.0), J.fill_(-1.0)
        timed(libs["this"], c, 1, stream)
        same = torch.equal(ref[0].view(torch.int64), T.view(torch.int64)) and torch.equal(ref[1].view(torch.int64), J.view(torch.int64))
        del ref
        torch.cuda.empty_cache()
        variants = {"parent": (libs["parent"], None), "this": (libs["this"], None)}
        report("%s  (outputs bitwise equal: %s)" % (title, same), alternate(variants, c, rounds, steps, stream))


if __name__ == "__main__":
    main()
