#!/usr/bin/env python
"""bench.py -- throughput of the Kinematics.jl hot path on B200 (driver contract in the task brief).

Default workload (BASELINE.json configs[1]): Fetch (data/fetch.urdf), 8 control joints, FP64, SoA:
    per configuration: get_transform for all 25 links + 6x8 geometric Jacobian of gripper_link,
    N = 2^24 random in-limit configurations per GPU (batch-sharded, weak scaling, no collective).
A "step" is one kin_eval over the whole batch (one kernel launch).  Inputs (1 GiB) and outputs
(46.7 GB) are far larger than the 126 MB L2, so nothing is served from cache between steps.

The same JSON line also carries
  * the north-star fused step (FK-all + gripper Jacobian + 16-sphere / fridge-SDF collision cost and gradient):
    `north_star` and, as flat scalars that survive the driver's record, `roofline.north_star_*`;
  * `e2e`: the same metric through kin_eval_host with pinned HOST buffers (copies inside the timed region), a plain
    pinned-copy probe taken on all ranks at once (`e2e.pcie_*`: the roofline of that path), the fused call and the two
    device-resident callers (batched IK, trajectory stack) end to end, each with its CPU baseline;
  * `small_batch`: kin_eval latency at the sizes the reference's solver callbacks really use (1, 10, 64, 1024).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the headline step returned in its last timed step (see dump_outputs) so that two builds can
be compared output for output: the inputs depend only on the arguments (seeded generators).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_LINKS, N_DOF, N_SPH = 25, 8, 16
# algorithmic bytes per configuration (SURVEY 8d / DESIGN.md): q in, 3x4 per link out, 6x8 Jacobian,
# S distances + S x n_dof gradients
BYTES_FKJ = 8 * N_DOF + 8 * 12 * N_LINKS + 8 * 6 * N_DOF                   # 2848
BYTES_COLL = 8 * N_DOF + 8 * N_SPH + 8 * N_SPH * N_DOF                      # 1216
BYTES_FUSED = BYTES_FKJ + 8 * N_SPH + 8 * N_SPH * N_DOF                     # 4000
METRIC = "fetch_fk_jacobian_configs_per_s"
UNIT = "configs/s"
WORKLOAD = "fk_all_links+gripper_jacobian"
WORKLOAD_FUSED = "fk_all_links+gripper_jacobian+collision_cost_grad(S=16,B=7,fd,reference-scratch)"


def base_config(world, n_per_gpu):
    """The `config` object: identical keys in the GPU arm and the reference arm."""
    return {"workload": WORKLOAD, "model": "data/fetch.urdf", "n_links": N_LINKS, "n_dof": N_DOF, "dtype": "f64",
            "configs_per_gpu": n_per_gpu, "layout": "soa", "parallelism": "batch-shard x%d, no collective" % world,
            "l2": "inputs+outputs per step (%.1f GB) exceed the 126 MB L2" % (BYTES_FKJ * n_per_gpu / 1e9)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_SAMPLE = 16384          # configurations written by --dump-outputs: T + J of the sample are 45.6 MB in float64


def dump_outputs(out_dir, T, J):
    """T.npy / J.npy: the columns of T (N_LINKS * 12 rows) and J (6 * N_DOF rows) of a fixed sample of the batch, in the
    SoA layout kin_eval writes them in (row-major: rows x sampled configurations, float64); sample_index.npy: the sampled
    configuration indices (ascending, stored as float64), drawn with seed 0."""
    import torch
    n = T.shape[1]
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    sel = torch.as_tensor(idx, device=T.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "T.npy"), T[:, sel].cpu().numpy())
    np.save(os.path.join(out_dir, "J.npy"), J[:, sel].cpu().numpy())
    np.save(os.path.join(out_dir, "sample_index.npy"), idx.astype(np.float64))


def ncu_traffic():
    """DRAM bytes per configuration from the committed `ncu --set full` captures (profiles/traffic.json, written by
    profiles/summarize.py); None when there is no capture of the kernel that is being timed."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 7 and r[3 + k].lower().startswith("active") for r in self.rows)]
        # the median under load: ignore idle samples (low power) when there are loaded ones
        loaded = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] if pw else sm
        return {"sm_mhz": float(np.median(loaded)) if loaded else None, "sm_max_mhz": mx[0] if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}


# ---------------------------------------------------------------------------------------------------
# CPU arms: the oracle port of the reference, all host threads, bounded samples.  (The only places where
# bench.py touches oracle/ and tests/scenes.py; the GPU arm never imports them.)
# ---------------------------------------------------------------------------------------------------
def _oracle_scene():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle import ref_model as R
    import scenes
    return R, scenes


def cpu_arm(workload, target_seconds, fused):
    """Times the restated reference CPU path (oracle/, kind = "port": the Julia reference cannot run here).
    Returns dict(value=configs/s, cores, sample, seconds)."""
    R, scenes = _oracle_scene()
    mo, jo, so = scenes.oracle_fetch(False)
    sdf_o = scenes.oracle_fridge_sdf() if fused else None
    threads = R.max_threads()
    links = mo.links[:N_LINKS]
    gl = R.find_link(mo, "gripper_link")

    def run(n, seed):
        q = scenes.random_configs(jo, n, False, seed=seed)
        t0 = time.perf_counter()
        R.batch_fused(so, jo, sdf_o, q, links, gl, with_rot=True, rpy_jac=False, n_threads=threads,
                      keep_outputs=False)
        return time.perf_counter() - t0

    run(20000, 1)                                   # warm-up (page-in, thread start)
    probe_n = 200000
    rate = probe_n / run(probe_n, 2)
    n = int(max(probe_n, min(rate * target_seconds, 5e7)))
    dt = run(n, 3)
    return {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d random in-limit Fetch configurations of the %s workload, one pass, %.1f s, %d pthreads, "
                      "one mechanism clone per thread" % (n, workload, dt, threads)}


def cpu_arm_trajectory_stack(target_seconds):
    """IneqConst stack of config 5 (planning.jl:55-68: per waypoint set_joint_angles + compute_coll_dists_and_grads!
    with truncation margin + 0.05) on all host threads: waypoint evaluations per second."""
    R, scenes = _oracle_scene()
    mo, jo, so = scenes.oracle_fetch(False)
    sdf_o = scenes.oracle_fridge_sdf()
    threads = R.max_threads()

    def run(n_prob, seed):
        rng = np.random.default_rng(seed)
        qs, qg = scenes.random_configs(jo, n_prob, False, seed=seed), scenes.random_configs(jo, n_prob, False, seed=seed + 1)
        X = qs[:, None, :] + (qg - qs)[:, None, :] * (np.arange(64) / 63.0)[None, :, None]      # planning.jl:304-308
        q = np.ascontiguousarray(X.reshape(-1, N_DOF))
        t0 = time.perf_counter()
        R.batch_collision(so, jo, sdf_o, q, 0.08, n_threads=threads)
        del rng
        return len(q), time.perf_counter() - t0

    run(64, 1)
    n, dt = run(1024, 2)
    n_prob = int(max(1024, min(4096 * 4, (n / dt) * target_seconds / 64)))
    n, dt = run(n_prob, 4)
    return {"value": n / dt, "unit": "waypoint_configs/s", "cores": threads, "kind": "port",
            "sample": "%d problems x 64 waypoints (margin 0.03, truncation 0.08, fridge SDF), %.1f s, %d pthreads" % (n_prob, dt, threads)}


def cpu_arm_ik(n_targets, collision=False):
    """inverse_kinematics! of the reference (SLSQP on f_objective with bounds; with ``collision`` the two-stage solve
    under IneqConst(margin 0.02) against the fridge, inverse_kinematics.jl:1-21) on every host core."""
    R, scenes = _oracle_scene()
    from oracle import callers_cpu as CC
    import scene_fetch
    mo, jo, so = scenes.oracle_fetch(False)
    q = scenes.random_configs(jo, (3 if collision else 1) * n_targets, False, seed=77)
    kw = {}
    if collision:      # targets = poses of configurations that clear the fridge by 0.03, as in the GPU row
        d, _, _ = R.batch_collision(so, jo, scenes.oracle_fridge_sdf(), q, with_grads=False)
        q = q[d.min(axis=1) > 0.03][:n_targets]
        kw = dict(sphere_fixture=os.path.join(ROOT, "data", "fetch_spheres.json"), obstacle_urdf=os.path.join(ROOT, "data", "fridge.urdf"),
                  obstacle_state=scene_fetch.FRIDGE_STATE, margin=0.02)
    Ts = R.batch_fk(mo, jo, q, [R.find_link(mo, "gripper_link")])[:, 0]
    procs = os.cpu_count() or 1
    r = CC.run_ik_baseline(os.path.join(ROOT, "data", "fetch.urdf"), scene_fetch.FETCH_JOINT_NAMES, "gripper_link", Ts,
                           np.array([0.2, 0, 0, 0, 0.5, 0, 0.5, 0]), with_rot=True, ftol=1e-10, n_procs=procs, **kw)
    out = {"value": r["targets_per_s"], "unit": "targets/s", "cores": r["procs"], "kind": "port",
           "fraction_objective_below_1e-6": r["fraction_objective_below_1e-6"], "mean_objective_evals": r["mean_evals"],
           "sample": "%d reachable gripper pose targets, scipy SLSQP (= the reference's SCIPY back-end; NLopt absent) driving the "
                     "oracle's C %s through ctypes (Python call overhead included), %d processes, %.1f s"
                     % (r["n"], "f_objective and IneqConst (two-stage solve, margin 0.02, fridge)" if collision else "f_objective",
                        r["procs"], r["seconds"])}
    if collision:
        out["fraction_reached_and_margin_kept"] = r["fraction_reached_and_margin_kept"]
    return out


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    vals, last = [], None
    per_step = max(2.0, min(20.0, 90.0 / max(1, args.steps + args.warmup)))
    for i in range(args.warmup + args.steps):
        last = cpu_arm(WORKLOAD, per_step, fused=False)
        if i >= args.warmup:
            vals.append(last["value"])
    v = float(np.mean(vals))
    cfg = base_config(args.gpus, args.n)
    cfg["note"] = "reference = CPU restatement of the Julia path (oracle/; Julia + scikit-robot are not installable here); " \
                  "each step is a bounded sample of the workload on all host threads"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": last["cores"], "kind": "port", "sample": last["sample"]},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--configs", dest="n", type=int, default=1 << 24, help="configurations per GPU")
    ap.add_argument("--configs-e2e", dest="n_e2e", type=int, default=1 << 21, help="configurations per e2e step (host buffers)")
    ap.add_argument("--skip-cpu", dest="no_cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--skip-north-star", dest="no_north_star", action="store_true")
    ap.add_argument("--skip-variants", dest="no_variants", action="store_true", help="skip the other BASELINE.md rows / layouts")
    ap.add_argument("--skip-callers", dest="no_callers", action="store_true", help="skip the IK / trajectory-stack rows")
    ap.add_argument("--skip-e2e", dest="no_e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a sample of the headline step's outputs as DIR/<name>.npy "
                                                          "(with --gpus > 1: rank 0's shard only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no outputs")
    if args.impl == "reference":
        return reference_main(args)

    import torch
    import kinematics_jl_b200 as K
    from kinematics_jl_b200 import lib as L
    from kinematics_jl_b200.device import device_model
    import scene_fetch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W = max(3, args.warmup)
    N = args.n
    dev = torch.device("cuda", local)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if dist is None:
            return float(x)
        t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def min_over_ranks(x):
        return -max_over_ranks(-float(x))

    # ---- model: Fetch + sphere fixture + fridge boxes (fridge_demo.jl:28) ----
    m, joints, sscc = scene_fetch.product_fetch(False)
    sdf = scene_fetch.product_fridge_sdf()
    K.set_joint_angles(m, joints, torch.zeros((1, N_DOF), dtype=torch.float64, device=dev))
    K.compute_coll_dists(sscc, joints, sdf)          # builds the device model and uploads sphere / box tables
    dm = device_model(m)
    lib = L.lib()

    # ---- synthetic inputs, resident in HBM (SoA: q[d][n]) ----
    g = torch.Generator(device=dev).manual_seed(rank)
    lo_np, hi_np = scene_fetch.joint_limits(joints)
    lo = torch.tensor(lo_np, device=dev, dtype=torch.float64)
    hi = torch.tensor(hi_np, device=dev, dtype=torch.float64)
    Q = lo[:, None] + (hi - lo)[:, None] * torch.rand((N_DOF, N), generator=g, device=dev, dtype=torch.float64)
    T = torch.empty((N_LINKS * 12, N), dtype=torch.float64, device=dev)
    J = torch.empty((6 * N_DOF, N), dtype=torch.float64, device=dev)
    fk_ids = np.arange(1, N_LINKS + 1, dtype=np.int32)
    gl = K.find_link(m, "gripper_link")
    jac_ids = np.array([gl.id], dtype=np.int32)
    ip = C.POINTER(C.c_int32)
    stream = torch.cuda.current_stream(dev)

    def make_call(n, q, T_, J_, V_=None, G_=None, layout=L.SOA):
        c = L.KinCall()
        c.precision, c.layout, c.n, c.q = L.F64, layout, n, q
        c.n_fk_links, c.fk_links, c.T_out = N_LINKS, fk_ids.ctypes.data_as(ip), T_
        c.n_jac_links, c.jac_links, c.J_out, c.with_rot = 1, jac_ids.ctypes.data_as(ip), J_, 1
        c.truncation_dist = float("inf")
        c.grad_mode, c.scratch_mode = L.GRAD_FD, L.SCRATCH_REFERENCE
        c.vals_out, c.grads_out = V_, G_
        c.stream = stream.cuda_stream
        return c

    def timed(call, steps, warm, model=None):
        h = (model or dm).h
        for _ in range(warm):
            L.check(lib.kin_eval(h, C.byref(call)))
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        n0 = lib.kin_launch_count()
        evs[0].record(stream)
        for i in range(steps):
            L.check(lib.kin_eval(h, C.byref(call)))
            evs[i + 1].record(stream)
        barrier()
        launches = lib.kin_launch_count() - n0
        total_ms = max_over_ranks(evs[0].elapsed_time(evs[-1]))
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        return total_ms, per, launches

    def launch_info(call, model=None):
        regs, smem, block, grid = (C.c_int32() for _ in range(4))
        L.check(lib.kin_query_launch((model or dm).h, C.byref(call), C.byref(regs), C.byref(smem), C.byref(block), C.byref(grid)))
        return {"regs": regs.value, "smem_bytes": smem.value, "block": block.value, "grid": grid.value}

    peak, peak_src = peaks()
    traffic = ncu_traffic()
    sampler = ClockSampler(local)

    # ---- headline: FK all links + gripper Jacobian ----
    call = make_call(N, Q.data_ptr(), T.data_ptr(), J.data_ptr())
    if rank == 0:
        sampler.start()
    total_ms, per, launches = timed(call, args.steps, W)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, T, J)           # before the variant rows below overwrite T / J
    ms_per_step = total_ms / args.steps
    value = world * N / (ms_per_step * 1e-3)
    kern_ms = float(np.mean(per))
    achieved = BYTES_FKJ * N / (kern_ms * 1e-3) / 1e9
    tr = traffic.get("fkj")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": tr["dram_bytes_per_config"] * N if tr else None,
                "traffic_source": tr["source"] if tr else None,
                "peak_source": peak_src, "kernel": (tr or {}).get("kernel", "kin_eval (FK + Jacobian)"),
                "algorithmic_bytes_per_config": BYTES_FKJ, "launch_ms": kern_ms}
    roofline.update({"launch_" + k: v for k, v in launch_info(call).items()})

    # ---- north star: fused FK-all + Jacobian + collision cost/grad ----
    north = None
    if not args.no_north_star:
        V = torch.empty((N_SPH, N), dtype=torch.float64, device=dev)
        G = torch.empty((N_SPH * N_DOF, N), dtype=torch.float64, device=dev)
        callf = make_call(N, Q.data_ptr(), T.data_ptr(), J.data_ptr(), V.data_ptr(), G.data_ptr())
        tms, perf_, _ = timed(callf, args.steps, W)
        ms_f = tms / args.steps
        ach_f = BYTES_FUSED * N / (float(np.mean(perf_)) * 1e-3) / 1e9
        trf = traffic.get("fused")
        north = {"workload": WORKLOAD_FUSED, "value": world * N / (ms_f * 1e-3), "unit": UNIT, "ms_per_step": ms_f,
                 "roofline": {"bound": "hbm-or-fp64 (see DESIGN.md)", "achieved": ach_f, "peak": peak, "unit": "GB/s",
                              "frac": ach_f / peak, "algorithmic_bytes_per_config": BYTES_FUSED,
                              "traffic": trf["dram_bytes_per_config"] * N if trf else None,
                              "fp64_pipe_frac_ncu": (trf or {}).get("fp64_pipe_frac"),
                              "kernel": (trf or {}).get("kernel"), "launch": launch_info(callf)}}
        # flat scalars inside a key the driver keeps (BENCH_r01 dropped the nested north_star object)
        roofline.update({"north_star_value": north["value"], "north_star_ms_per_step": ms_f,
                         "north_star_frac": ach_f / peak, "north_star_bytes_per_config": BYTES_FUSED,
                         "north_star_fp64_pipe_frac_ncu": (trf or {}).get("fp64_pipe_frac"),
                         "north_star_block": north["roofline"]["launch"]["block"]})
        del V, G

    # ---- other rows of BASELINE.md section 3, same batch (reported, not the headline) ----
    variants = {}
    if not args.no_variants:
        def variant(name, bytes_per_cfg, call_, n_=N, model=None):
            tms_, per_, _ = timed(call_, max(3, args.steps // 2), W, model)
            ms_ = float(np.mean(per_))
            variants[name] = {"value": world * n_ / (ms_ * 1e-3), "unit": UNIT, "ms_per_step": ms_, "configs": n_,
                              "algorithmic_bytes_per_config": bytes_per_cfg,
                              "hbm_frac": bytes_per_cfg * n_ / (ms_ * 1e-3) / 1e9 / peak, "launch": launch_info(call_, model)}
        cg = make_call(N, Q.data_ptr(), T.data_ptr(), J.data_ptr())
        cg.n_fk_links, cg.fk_links = 1, jac_ids.ctypes.data_as(ip)
        variant("fk_gripper+gripper_jacobian", 8 * N_DOF + 96 + 384, cg)
        V = torch.empty((N_SPH, N), dtype=torch.float64, device=dev)
        G = torch.empty((N_SPH * N_DOF, N), dtype=torch.float64, device=dev)
        cc = make_call(N, Q.data_ptr(), None, None, V.data_ptr(), G.data_ptr())
        cc.n_fk_links = cc.n_jac_links = 0
        variant("collision_cost_grad(S=16,B=7,fd,reference-scratch)", BYTES_COLL, cc)
        cc2 = make_call(N, Q.data_ptr(), None, None, V.data_ptr(), G.data_ptr())
        cc2.n_fk_links = cc2.n_jac_links = 0
        cc2.grad_mode, cc2.scratch_mode = L.GRAD_ANALYTIC, L.SCRATCH_CLEAN
        variant("collision_cost_grad(S=16,B=7,analytic,clean-scratch)", BYTES_COLL, cc2)
        del V, G
        # distances only (compute_coll_dists!, collision.jl:51-58) and their per-configuration reductions
        # (kin_collision_summary: min distance / sphere / hinge cost -- a collision CHECK; 20 B out per configuration)
        dmin_ = torch.empty(N, dtype=torch.float64, device=dev)
        cost_ = torch.empty(N, dtype=torch.float64, device=dev)
        amin_ = torch.empty(N, dtype=torch.int32, device=dev)

        def summary():
            L.check(lib.kin_collision_summary(dm.h, L.F64, L.SOA, Q.data_ptr(), N, 0.03, dmin_.data_ptr(), amin_.data_ptr(),
                                              cost_.data_ptr(), stream.cuda_stream))
        for _ in range(W):
            summary()
        barrier()
        s_steps = max(3, args.steps // 2)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(s_steps):
            summary()
        ev1.record(stream)
        barrier()
        ms_ = max_over_ranks(ev0.elapsed_time(ev1)) / s_steps
        variants["collision_check_summary(min distance, argmin sphere, hinge cost)"] = {
            "value": world * N / (ms_ * 1e-3), "unit": UNIT, "ms_per_step": ms_, "configs": N,
            "algorithmic_bytes_per_config": 8 * N_DOF + 20, "note": "compute-bound: 16 spheres x 7 boxes per configuration, 84 B of I/O",
            "fraction_in_collision": float((dmin_ < 0).double().mean())}
        del dmin_, cost_, amin_
        # the tiled (AoSoA-32) layout: one contiguous block per warp
        Qt = Q.t().reshape(N // 32, 32, N_DOF).permute(0, 2, 1).contiguous()
        Tt = torch.empty((N // 32, N_LINKS * 12, 32), dtype=torch.float64, device=dev)
        Jt = torch.empty((N // 32, 6 * N_DOF, 32), dtype=torch.float64, device=dev)
        ct = make_call(N, Qt.data_ptr(), Tt.data_ptr(), Jt.data_ptr(), layout=L.TILED32)
        variant("fk_all_links+gripper_jacobian_tiled32_layout", BYTES_FKJ, ct)
        Vt = torch.empty((N // 32, N_SPH, 32), dtype=torch.float64, device=dev)
        Gt = torch.empty((N // 32, N_SPH * N_DOF, 32), dtype=torch.float64, device=dev)
        ctf = make_call(N, Qt.data_ptr(), Tt.data_ptr(), Jt.data_ptr(), Vt.data_ptr(), Gt.data_ptr(), layout=L.TILED32)
        variant("fused_tiled32_layout", BYTES_FUSED, ctf)
        del Qt, Tt, Jt, Vt, Gt
        # the optional FP32 mode (1e-5 tolerance), fused step, SoA
        Q32 = Q.float()
        T32 = torch.empty((N_LINKS * 12, N), dtype=torch.float32, device=dev)
        J32 = torch.empty((6 * N_DOF, N), dtype=torch.float32, device=dev)
        V32 = torch.empty((N_SPH, N), dtype=torch.float32, device=dev)
        G32 = torch.empty((N_SPH * N_DOF, N), dtype=torch.float32, device=dev)
        c32 = make_call(N, Q32.data_ptr(), T32.data_ptr(), J32.data_ptr(), V32.data_ptr(), G32.data_ptr())
        c32.precision = L.F32
        c32.grad_mode = L.GRAD_ANALYTIC          # a 1e-7 forward difference is meaningless in FP32
        variant("fused_fp32_mode(analytic gradient)", BYTES_FUSED // 2, c32)
        del Q32, T32, J32, V32, G32
        # the fused step in the AoS layout (one contiguous record per configuration, planning.jl:58)
        Na = min(N, 1 << 22)
        Qa = Q[:, :Na].t().contiguous()
        Ta = torch.empty((Na, N_LINKS * 12), dtype=torch.float64, device=dev)
        Ja = torch.empty((Na, 6 * N_DOF), dtype=torch.float64, device=dev)
        Va = torch.empty((Na, N_SPH), dtype=torch.float64, device=dev)
        Ga = torch.empty((Na, N_SPH * N_DOF), dtype=torch.float64, device=dev)
        ca = make_call(Na, Qa.data_ptr(), Ta.data_ptr(), Ja.data_ptr(), Va.data_ptr(), Ga.data_ptr(), layout=L.AOS)
        variant("fused_aos_layout", BYTES_FUSED, ca, Na)
        del Qa, Ta, Ja, Va, Ga
        # the fused step on the Fetch WITH the planar base (11 columns: SURVEY 8d variant), SoA
        mb, jb, sb = scene_fetch.product_fetch(True)
        Nb = min(N, 1 << 22)
        K.set_joint_angles(mb, jb, torch.zeros((1, N_DOF + 3), dtype=torch.float64, device=dev))
        K.compute_coll_dists(sb, jb, sdf)
        dmb = device_model(mb)
        gb = torch.Generator(device=dev).manual_seed(1000 + rank)
        lob = torch.cat([lo, torch.tensor([-1.0, -1.0, -np.pi], device=dev, dtype=torch.float64)])
        hib = torch.cat([hi, torch.tensor([1.0, 1.0, np.pi], device=dev, dtype=torch.float64)])
        Qb = lob[:, None] + (hib - lob)[:, None] * torch.rand((N_DOF + 3, Nb), generator=gb, device=dev, dtype=torch.float64)
        Tb = torch.empty((N_LINKS * 12, Nb), dtype=torch.float64, device=dev)
        Jb = torch.empty((6 * (N_DOF + 3), Nb), dtype=torch.float64, device=dev)
        Vb = torch.empty((N_SPH, Nb), dtype=torch.float64, device=dev)
        Gb = torch.empty((N_SPH * (N_DOF + 3), Nb), dtype=torch.float64, device=dev)
        cb = make_call(Nb, Qb.data_ptr(), Tb.data_ptr(), Jb.data_ptr(), Vb.data_ptr(), Gb.data_ptr())
        jac_b = np.array([K.find_link(mb, "gripper_link").id], dtype=np.int32)
        cb.jac_links = jac_b.ctypes.data_as(ip)
        bytes_b = 8 * (N_DOF + 3) + 8 * 12 * N_LINKS + 8 * 6 * (N_DOF + 3) + 8 * N_SPH + 8 * N_SPH * (N_DOF + 3)
        variant("fused_with_planar_base(11 columns)", bytes_b, cb, Nb, dmb)
        del Qb, Tb, Jb, Vb, Gb
        # a dual-arm mechanism with the planar base (data/dual_arm.urdf: 18 columns, 37 links, 19 spheres, 3 boxes -- the size
        # class of the PR2 of fridge_demo.jl): FK of all links + collision cost / gradient, SoA.  Above 16 columns the
        # specialised kernel takes the launch shape with the most threads per SM whose shared scratch fits (DESIGN 7, round 2d)
        md, jd, sd, sdfd = scene_fetch.product_dual_arm(True)
        ndd, nld, nsd, Nd = len(jd) + 3, len(md.links), len(sd.sphere_radii), min(N, 1 << 21)
        K.set_joint_angles(md, jd, torch.zeros((1, ndd), dtype=torch.float64, device=dev))
        K.compute_coll_dists(sd, jd, sdfd)
        dmd = device_model(md)
        gd = torch.Generator(device=dev).manual_seed(2000 + rank)
        Qd = 2.0 * torch.rand((ndd, Nd), generator=gd, device=dev, dtype=torch.float64) - 1.0
        Td = torch.empty((nld * 12, Nd), dtype=torch.float64, device=dev)
        Vd = torch.empty((nsd, Nd), dtype=torch.float64, device=dev)
        Gd = torch.empty((nsd * ndd, Nd), dtype=torch.float64, device=dev)
        fk_d = np.array([l.id for l in md.links], dtype=np.int32)
        cd = make_call(Nd, Qd.data_ptr(), Td.data_ptr(), None, Vd.data_ptr(), Gd.data_ptr())
        cd.n_fk_links, cd.fk_links, cd.n_jac_links, cd.jac_links = nld, fk_d.ctypes.data_as(ip), 0, None
        variant("dual_arm_with_planar_base(18 columns,37 links,S=19,B=3):fk_all_links+collision_cost_grad", 8 * (ndd + 12 * nld + nsd + nsd * ndd), cd, Nd, dmd)
        del Qd, Td, Vd, Gd

    # ---- small batches: the sizes the reference's solver callbacks really evaluate (one configuration per IK
    #      iteration, n_wp = 10..64 per planning iteration): latency of one fused kin_eval, launch to completion ----
    small = {}
    if not args.no_variants:
        small["note"] = "fused kin_eval (FK all links + gripper Jacobian + collision cost / gradient) of n configurations; after a few small " \
                        "calls the library switches to the specialised kernel of this program (negative block size)"
        ld_s = 1024
        Qs_ = Q[:, :ld_s].contiguous()
        Ts_ = torch.empty((N_LINKS * 12, ld_s), dtype=torch.float64, device=dev)
        Js_ = torch.empty((6 * N_DOF, ld_s), dtype=torch.float64, device=dev)
        Vs = torch.empty((N_SPH, ld_s), dtype=torch.float64, device=dev)
        Gs = torch.empty((N_SPH * N_DOF, ld_s), dtype=torch.float64, device=dev)
        for n_s in (1, 10, 64, 1024):
            cs = make_call(n_s, Qs_.data_ptr(), Ts_.data_ptr(), Js_.data_ptr(), Vs.data_ptr(), Gs.data_ptr())
            cs.batch_stride = ld_s
            for _ in range(20):
                L.check(lib.kin_eval(dm.h, C.byref(cs)))
            torch.cuda.synchronize(dev)
            reps = 200
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            a.record(stream)
            for _ in range(reps):
                L.check(lib.kin_eval(dm.h, C.byref(cs)))
            b.record(stream)
            t_issue = time.perf_counter() - t0
            torch.cuda.synchronize(dev)
            # one call + synchronise: what a solver callback that needs the numbers on the host waits for
            t0 = time.perf_counter()
            for _ in range(50):
                L.check(lib.kin_eval(dm.h, C.byref(cs)))
                torch.cuda.synchronize(dev)
            t_sync = (time.perf_counter() - t0) / 50
            small["n=%d" % n_s] = {"device_us_per_call_back_to_back": 1e3 * a.elapsed_time(b) / reps,
                               "host_issue_us_per_call": 1e6 * t_issue / reps, "call_plus_sync_us": 1e6 * t_sync,
                               "launch": launch_info(cs)}
        del Vs, Gs, Qs_, Ts_, Js_

    # ---- configs 4 and 5 of BASELINE.json (caller-side rows of SURVEY 8f), through the host mirror ----
    callers = {}
    if not args.no_callers:
        def ev_time(fn, reps):
            fn()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(reps):
                r = fn()
            b.record(stream)
            torch.cuda.synchronize(dev)
            return max_over_ranks(a.elapsed_time(b) / reps), r
        # config 5: 4096 problems x 64 waypoints, straight-line initial trajectories, IneqConst stack
        # (margin 0.03, truncation 0.08), problems sharded over the ranks, stacked outputs all-gathered
        P, n_wp = 4096, 64
        p0, p1 = K.shard_range(P, rank, world)
        gq = torch.Generator(device=dev).manual_seed(1234)
        qs = lo + (hi - lo) * torch.rand((P, N_DOF), generator=gq, device=dev, dtype=torch.float64)
        qg = lo + (hi - lo) * torch.rand((P, N_DOF), generator=gq, device=dev, dtype=torch.float64)
        X = K.create_straight_trajectory(qs[p0:p1], qg[p0:p1], n_wp)
        G5 = K.IneqConst(sscc, joints, sdf, n_wp, 0.03)
        ms_eval, (v5, g5) = ev_time(lambda: G5(X), 5)
        slab5 = torch.empty((N_SPH + N_SPH * N_DOF, (p1 - p0) * n_wp), dtype=torch.float64, device=dev)
        out5 = torch.empty((world,) + tuple(slab5.shape), dtype=torch.float64, device=dev) if world > 1 else None
        # the kernel writes [vals | grads] straight into one slab, which one all_gather_into_tensor distributes
        ms_all, _ = ev_time(lambda: K.gather_packed(G5.evaluate_packed(X, slab5)[0], n_wp, N_DOF, N_SPH, out=out5), 5)
        row5 = {"waypoint_configs_per_s_eval_only": P * n_wp / (ms_eval * 1e-3), "waypoint_configs_per_s_with_allgather": P * n_wp / (ms_all * 1e-3),
                "ms_eval": ms_eval, "ms_eval_plus_allgather": ms_all, "n_gpus": world,
                "gathered_bytes": 8 * P * n_wp * (N_SPH + N_SPH * N_DOF),
                "collective": "NCCL all_gather_into_tensor of one packed [vals | grads] slab" if world > 1 else "none (1 rank)"}
        # end to end: xi from pinned host memory, values + block-diagonal Jacobian back to pinned host memory
        if not args.no_e2e:
            Xh = torch.empty(X.shape, dtype=torch.float64).pin_memory()
            Xh.copy_(X)
            vh = torch.empty(v5.shape, dtype=torch.float64).pin_memory()
            gh = torch.empty(g5.shape, dtype=torch.float64).pin_memory()

            def traj_e2e():
                Xd = Xh.to(dev, non_blocking=True)
                v_, g_ = G5(Xd)
                vh.copy_(v_, non_blocking=True)
                gh.copy_(g_, non_blocking=True)
                torch.cuda.synchronize(dev)
            traj_e2e()
            barrier()
            t0 = time.perf_counter()
            for _ in range(5):
                traj_e2e()
            dt5 = max_over_ranks((time.perf_counter() - t0) / 5)
            row5["e2e_waypoint_configs_per_s"] = P * n_wp / dt5
            row5["e2e_h2d_bytes"] = Xh.numel() * 8
            row5["e2e_d2h_bytes"] = (vh.numel() + gh.numel()) * 8
            row5["e2e_check_max_abs_diff_vs_device"] = float((vh.to(dev) - v5).abs().max())
            del Xh, vh, gh
        callers["trajectory_stack(4096x64)"] = row5
        del X, v5, g5, slab5, out5
        # config 4: 2^20 independent gripper pose targets (FK of random in-limit configurations)
        Nik = 1 << 20
        qt = lo + (hi - lo) * torch.rand((Nik, N_DOF), generator=gq, device=dev, dtype=torch.float64)
        K.set_joint_angles(m, joints, qt)
        Tg = K.get_transform(m, gl)
        yaw = torch.atan2(Tg[:, 1, 0], Tg[:, 0, 0])
        c1, s1 = torch.cos(yaw), torch.sin(yaw)
        pitch = torch.atan2(-Tg[:, 2, 0], torch.sqrt(Tg[:, 2, 1] ** 2 + Tg[:, 2, 2] ** 2))
        roll = torch.atan2(Tg[:, 0, 2] * s1 - Tg[:, 1, 2] * c1, Tg[:, 1, 1] * c1 - Tg[:, 0, 1] * s1)
        tg = torch.cat([Tg[:, :, 3], roll[:, None], pitch[:, None], yaw[:, None]], dim=1).contiguous()
        q0 = torch.tensor([0.2, 0, 0, 0, 0.5, 0, 0.5, 0], device=dev, dtype=torch.float64).repeat(Nik, 1)
        K.set_joint_angles(m, joints, q0)
        ms_it, _ = ev_time(lambda: K.pose_constraint(m, gl, joints, tg, True), 5)
        # warm-up at the measured size: builds the kernel and grows the stream-ordered pools / the allocator's blocks
        K.inverse_kinematics_batch(m, gl, joints, tg, q0, with_rot=True, iters=40, restarts=2)
        barrier()
        t0 = time.perf_counter()
        qsol, fsol = K.inverse_kinematics_batch(m, gl, joints, tg, q0, with_rot=True, iters=40)
        torch.cuda.synchronize(dev)
        t_single = max_over_ranks(time.perf_counter() - t0)
        ok_single = float((fsol < 1e-6).double().mean())
        barrier()
        t0 = time.perf_counter()
        qsol, fsol = K.inverse_kinematics_batch(m, gl, joints, tg, q0, with_rot=True, iters=40, restarts=2)
        torch.cuda.synchronize(dev)
        t_solve = max_over_ranks(time.perf_counter() - t0)
        K.set_joint_angles(m, joints, qsol)
        vv, _ = K.pose_constraint(m, gl, joints, tg, True)
        vv[:, 3:] = torch.remainder(vv[:, 3:] + np.pi, 2 * np.pi) - np.pi
        ok = float((vv.abs().amax(dim=1) < 1e-3).double().mean())
        row4 = {"residual_and_jacobian_evals_per_s": world * Nik / (ms_it * 1e-3), "ms_per_evaluation": ms_it,
                "solver": "kin_ik_solve: device-resident Levenberg-Marquardt, 40 iterations per solve in stages of 3, 4, 6, 9 and 18 "
                          "iterations over the still-running problems (index list compacted between stages, 8 bytes read back); "
                          "problems above the tolerance are re-seeded twice",
                "solve_seconds_one_solve": t_single, "fraction_f_below_1e-6_one_solve": ok_single,
                "solve_seconds_with_2_restarts": t_solve, "targets_per_s": world * Nik / t_solve,
                "solve_over_40_evaluations": t_solve / (40 * ms_it * 1e-3), "fraction_within_1e-3": ok, "n_gpus": world}
        if not args.no_e2e:
            tgh = torch.empty(tg.shape, dtype=torch.float64).pin_memory()
            tgh.copy_(tg)
            qh_ = torch.empty(qsol.shape, dtype=torch.float64).pin_memory()
            barrier()
            t0 = time.perf_counter()
            tgd = tgh.to(dev, non_blocking=True)
            q_e, _ = K.inverse_kinematics_batch(m, gl, joints, tgd, q0, with_rot=True, iters=40, restarts=2)
            qh_.copy_(q_e, non_blocking=True)
            torch.cuda.synchronize(dev)
            dt4 = max_over_ranks(time.perf_counter() - t0)
            row4["e2e_targets_per_s"] = world * Nik / dt4
            row4["e2e_h2d_bytes"] = tgh.numel() * 8
            row4["e2e_d2h_bytes"] = qh_.numel() * 8
            row4["e2e_check_max_abs_diff_vs_device"] = float((qh_.to(dev) - qsol).abs().max())
            del tgh, qh_
        callers["batched_ik(2^20 targets)"] = row4
        # config 4 proper: the same targets under the reference's hard collision constraint (inverse_kinematics.jl:14-19,
        # dists - 0.02 >= 0 against the fridge), targets restricted to poses of configurations that clear the fridge by 0.03
        K.set_joint_angles(m, joints, qt)
        feas = torch.nonzero(K.compute_coll_dists(sscc, joints, sdf).amin(dim=1) > 0.03).squeeze(1)
        tgc, q0c = tg[feas].contiguous(), q0[feas].contiguous()
        Nc = int(feas.numel())
        K.inverse_kinematics_batch(m, gl, joints, tgc, q0c, with_rot=True, iters=40, sscc=sscc, sdf=sdf, coll_iters=2)   # warm-up (builds the large-batch kernels, grows the workspace pool)
        torch.cuda.synchronize(dev)
        barrier()
        t0 = time.perf_counter()
        qc_, fc_, dc_ = K.inverse_kinematics_batch(m, gl, joints, tgc, q0c, with_rot=True, iters=40, sscc=sscc, sdf=sdf, margin=0.02,
                                                   coll_iters=60, return_dmin=True)
        torch.cuda.synchronize(dev)
        t_c1 = max_over_ranks(time.perf_counter() - t0)
        ok_c1 = float(((fc_ <= 1e-6) & (dc_ >= 0.02 - 1e-5)).double().mean())
        barrier()
        t0 = time.perf_counter()
        qc_, fc_, dc_ = K.inverse_kinematics_batch(m, gl, joints, tgc, q0c, with_rot=True, iters=40, sscc=sscc, sdf=sdf, margin=0.02,
                                                   coll_iters=60, restarts=2, return_dmin=True)
        torch.cuda.synchronize(dev)
        t_c2 = max_over_ranks(time.perf_counter() - t0)
        ok_c2 = float(((fc_ <= 1e-6) & (dc_ >= 0.02 - 1e-5)).double().mean())
        callers["batched_ik_collision_constrained"] = {
            "targets": Nc, "n_gpus": world,
            "solver": "kin_ik_solve: pose-only warm start (one launch) + augmented-Lagrangian LM under dists - 0.02 >= 0 vs the fridge "
                      "(one fused kin_eval + one step kernel per iteration over the still-running problems: active list re-compacted at iterations 1, 2, 3, 4, 6, 8, 12, ..., 8 bytes read back each time; 61 pairs at most)",
            "solve_seconds_one_seed": t_c1, "fraction_reached_and_margin_kept_one_seed": ok_c1,
            "solve_seconds_with_2_restarts": t_c2, "fraction_reached_and_margin_kept": ok_c2,
            "targets_per_s": world * Nc / t_c2, "min_distance_over_batch": float(dc_.min())}
        del qt, Tg, tg, q0, qsol, fsol, vv, tgc, q0c, qc_, fc_, dc_, feas
        K.set_joint_angles(m, joints, torch.zeros((1, N_DOF), dtype=torch.float64, device=dev))

    # ---- e2e: the C-ABI call with HOST buffers (pinned), H2D + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        Ne = min(args.n_e2e, N)
        qh = torch.empty((N_DOF, Ne), dtype=torch.float64).pin_memory()
        qh.copy_(Q[:, :Ne].cpu())
        Th = torch.empty((N_LINKS * 12, Ne), dtype=torch.float64).pin_memory()
        Jh = torch.empty((6 * N_DOF, Ne), dtype=torch.float64).pin_memory()
        Th.fill_(-1.0)
        calle = make_call(Ne, qh.data_ptr(), Th.data_ptr(), Jh.data_ptr())

        def host_loop(call_, steps):
            for _ in range(2):
                L.check(lib.kin_eval_host(dm.h, C.byref(call_)))
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                L.check(lib.kin_eval_host(dm.h, C.byref(call_)))     # returns when the outputs are in host memory
            return max_over_ranks(time.perf_counter() - t0)
        def transfer_counters():
            v = [C.c_int64() for _ in range(3)]
            L.check(lib.kin_host_transfer_bytes(*[C.byref(x) for x in v]))
            return [x.value for x in v]
        e_steps = max(3, min(args.steps, 10))
        # (a) every output row over PCIe (what round 1 measured); (b) the default: rows of T / J that do not depend on
        # the configuration are written by host threads instead of crossing PCIe (kin_b200.h: kin_eval_host)
        os.environ["KIN_HOST_NO_CONST_FILL"] = "1"
        e_dt_all = host_loop(calle, e_steps)
        del os.environ["KIN_HOST_NO_CONST_FILL"]
        Th.fill_(-1.0)
        Jh.fill_(-1.0)
        c0 = transfer_counters()
        e_dt = host_loop(calle, e_steps)
        c1 = transfer_counters()
        h2d_b, d2h_b, fill_b = [(b - a) // (e_steps + 2) for a, b in zip(c0, c1)]       # host_loop makes 2 warm-up calls
        # the check depends on the copies AND on the host-side fill: every row of T and J of the LAST configuration and of
        # one in the middle, host result vs the device-resident result of the same inputs (T / J of the headline run)
        gcol = 12 * (gl.id - 1) + 9
        cols = sorted({i for i in (0, Ne - 1, Ne // 2, Ne // 3 + 17, (1 << 17) - 1, 1 << 17) if 0 <= i < Ne})   # incl. both sides of a staging-chunk boundary
        L.check(lib.kin_eval(dm.h, C.byref(call)))          # the variant rows above reuse T / J: regenerate the headline outputs
        torch.cuda.synchronize(dev)
        by_col = {i: (float((Th[:, i] - T[:, i].cpu()).abs().max()), float((Jh[:, i] - J[:, i].cpu()).abs().max())) for i in cols}
        dT, dJ = max(v[0] for v in by_col.values()), max(v[1] for v in by_col.values())
        if max(dT, dJ) > 0:
            sys.stderr.write("e2e check: host result differs from the device result, (max |dT|, max |dJ|) by column: %r\n" % by_col)
            for i in cols:
                rows_bad = torch.nonzero((Th[:, i] - T[:, i].cpu()).abs() > 0).flatten().tolist()
                sys.stderr.write("  column %d: T rows %r\n" % (i, rows_bad[:40]))
        e2e = {"value": world * Ne * e_steps / e_dt, "unit": UNIT, "h2d_bytes_per_step": h2d_b,
               "d2h_bytes_per_step": d2h_b, "host_filled_bytes_per_step": fill_b, "configs_per_step": Ne, "steps": e_steps,
               "api": "kin_eval_host (C ABI, pinned host q / T / J, chunked H2D -> kernel -> D2H on 3 streams; %d of the %d output "
                      "rows do not cross PCIe: rows that do not depend on the configuration are filled, and rows that hold the "
                      "same value as another row (+-) are copied, by host threads)"
                      % (fill_b // (8 * Ne), N_LINKS * 12 + 6 * N_DOF),
               "value_all_rows_over_pcie": world * Ne * e_steps / e_dt_all,
               "check": float(Th[gcol, Ne - 1]), "check_max_abs_diff_vs_device": float(max(dT, dJ)),
               "gbs_per_gpu": (d2h_b + h2d_b) * e_steps / e_dt / 1e9}
        # PCIe roofline of that path: a plain pinned D2H / H2D copy of 1 GiB, on all ranks AT THE SAME TIME
        probe_bytes = 1 << 30
        ph = torch.empty(probe_bytes // 8, dtype=torch.float64).pin_memory()
        pd = torch.empty(probe_bytes // 8, dtype=torch.float64, device=dev)

        def copy_gbs(dst, src):
            dst.copy_(src, non_blocking=True)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            b.record(stream)
            torch.cuda.synchronize(dev)
            return 4 * probe_bytes / (a.elapsed_time(b) * 1e-3) / 1e9
        d2h = copy_gbs(ph, pd)
        h2d = copy_gbs(pd, ph)
        e2e["pcie_d2h_gbs_per_gpu_min_over_ranks"] = min_over_ranks(d2h)
        e2e["pcie_h2d_gbs_per_gpu_min_over_ranks"] = min_over_ranks(h2d)
        e2e["pcie_peak_gbs"] = e2e["pcie_d2h_gbs_per_gpu_min_over_ranks"]
        e2e["pcie_frac"] = (e2e["gbs_per_gpu"]) / e2e["pcie_peak_gbs"]
        e2e["pcie_note"] = "peak = plain cudaMemcpyAsync D2H of 1 GiB pinned, all %d ranks concurrently; the path moves %d B " \
                           "of results per configuration over PCIe (%d B with every row copied)" \
                           % (world, d2h_b // Ne, 8 * (N_LINKS * 12 + 6 * N_DOF))
        del ph, pd
        # the fused north-star call end to end (3936 B of results per configuration)
        if not args.no_north_star:
            Vh = torch.empty((N_SPH, Ne), dtype=torch.float64).pin_memory()
            Gh = torch.empty((N_SPH * N_DOF, Ne), dtype=torch.float64).pin_memory()
            callfe = make_call(Ne, qh.data_ptr(), Th.data_ptr(), Jh.data_ptr(), Vh.data_ptr(), Gh.data_ptr())
            f_steps = max(3, e_steps // 2)
            f_dt = host_loop(callfe, f_steps)
            e2e["north_star_value"] = world * Ne * f_steps / f_dt
            e2e["north_star_d2h_bytes_per_step"] = d2h_b + 8 * (N_SPH + N_SPH * N_DOF) * Ne
            e2e["north_star_pcie_frac"] = (e2e["north_star_d2h_bytes_per_step"] + h2d_b) * f_steps / f_dt / 1e9 / e2e["pcie_peak_gbs"]
            del Vh, Gh
        for name, row, key in (("ik", callers.get("batched_ik(2^20 targets)"), "e2e_targets_per_s"),
                               ("trajectory_stack", callers.get("trajectory_stack(4096x64)"), "e2e_waypoint_configs_per_s")):
            if row and key in row:
                e2e[name + "_" + key] = row[key]
        del qh, Th, Jh

    # ---- CPU baselines (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_arm(WORKLOAD, 12.0, fused=False)
        if north is not None:
            north["cpu_baseline"] = cpu_arm(WORKLOAD_FUSED, 10.0, fused=True)
            roofline["north_star_cpu_baseline_value"] = north["cpu_baseline"]["value"]
            if e2e is not None and "north_star_value" in e2e:
                e2e["north_star_cpu_baseline_value"] = north["cpu_baseline"]["value"]
        if callers:
            c5 = cpu_arm_trajectory_stack(6.0)
            callers["trajectory_stack(4096x64)"]["cpu_baseline"] = c5
            c4 = cpu_arm_ik(64 * (os.cpu_count() or 1))
            callers["batched_ik(2^20 targets)"]["cpu_baseline"] = c4
            callers["batched_ik_collision_constrained"]["cpu_baseline"] = cpu_arm_ik(16 * (os.cpu_count() or 1), collision=True)
            if e2e is not None:
                e2e["trajectory_stack_cpu_baseline_value"] = c5["value"]
                e2e["ik_cpu_baseline_value"] = c4["value"]

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "gpu_launches": int(launches),
                "config": base_config(world, N), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
                "north_star": north, "variants": variants, "small_batch": small, "callers": callers}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
