"""ctypes binding of libkin_b200.so (include/kin_b200.h).  There is NO fallback: if the shared
library is missing or there is no CUDA device, every operator raises."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "libkin_b200.so")
SO_PATH_DEBUG = os.path.join(HERE, "libkin_b200_debug.so")
CSRC = os.path.join(HERE, "csrc")

F64, F32 = 0, 1
SOA, AOS, TILED32 = 0, 1, 2
FIXED, REVOLUTE, PRISMATIC = 0, 1, 2
GRAD_FD, GRAD_ANALYTIC, GRAD_FD_DIRECT = 0, 1, 2
PRIM_BOX, PRIM_SPHERE, PRIM_CYLINDER, PRIM_GRID = 0, 1, 2, 3
MAX_GRID_VALUES = 1 << 28
SCRATCH_REFERENCE, SCRATCH_CLEAN = 0, 1
POSE_IK_OBJECTIVE, POSE_CONSTRAINT = 0, 1

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "-cudart", "static"]
SOURCES = ["kin_b200.cu", "kin_model.cpp", "kin_codegen.cpp", "kin_jit.cpp"]
EMBEDDED = ["kin_device_math.cuh", "kin_gen_skeleton.cuh"]      # linked in as text for NVRTC (kin_jit.cpp)


class KinError(RuntimeError):
    pass


class KinModelDesc(C.Structure):
    _fields_ = [("n_links", C.c_int32), ("parent_link", _ip), ("joint_type", _ip), ("joint_pose", _dp),
                ("joint_axis", _dp), ("q_index", _ip), ("default_angle", _dp), ("n_joints", C.c_int32),
                ("with_base", C.c_int32), ("n_spheres", C.c_int32), ("sphere_link", _ip), ("sphere_center", _dp),
                ("sphere_radius", _dp), ("n_boxes", C.c_int32), ("box_pose", _dp), ("box_width", _dp)]


class KinCall(C.Structure):
    _fields_ = [("precision", C.c_int32), ("layout", C.c_int32), ("n", C.c_int64), ("batch_stride", C.c_int64),
                ("q", C.c_void_p),
                ("n_fk_links", C.c_int32), ("fk_links", _ip), ("T_out", C.c_void_p),
                ("n_jac_links", C.c_int32), ("jac_links", _ip), ("with_rot", C.c_int32), ("rpy_jac", C.c_int32),
                ("keep_irrelevant", C.c_int32), ("J_out", C.c_void_p),
                ("truncation_dist", C.c_double), ("grad_mode", C.c_int32), ("scratch_mode", C.c_int32),
                ("vals_out", C.c_void_p), ("grads_out", C.c_void_p), ("argmin_out", C.c_void_p),
                ("vals_offset", C.c_double), ("stream", C.c_void_p)]


class KinIkCall(C.Structure):
    _fields_ = [("n", C.c_int64), ("link_id", C.c_int32), ("with_rot", C.c_int32), ("iters", C.c_int32), ("ftol", C.c_double),
                ("lambda0", C.c_double), ("targets", C.c_void_p), ("q0", C.c_void_p), ("lower", _dp), ("upper", _dp),
                ("q_out", C.c_void_p), ("f_out", C.c_void_p), ("iters_out", C.c_void_p), ("stream", C.c_void_p),
                ("collision", C.c_int32), ("reserved_", C.c_int32), ("margin", C.c_double), ("coll_weight", C.c_double),
                ("ctol", C.c_double), ("dmin_out", C.c_void_p)]


ERR_UNAVAILABLE = -6

EXPORTS = ["kin_last_error", "kin_abi_version", "kin_build_id", "kin_debug_build", "kin_model_create", "kin_model_destroy", "kin_model_set_spheres",
           "kin_model_set_boxes", "kin_model_set_primitives", "kin_sdf_points_prims", "kin_collision_summary", "kin_model_n_dof", "kin_model_n_spheres", "kin_model_n_boxes", "kin_eval",
           "kin_eval_host", "kin_fk_links", "kin_fk_jacobian", "kin_collision", "kin_launch_count",
           "kin_query_launch", "kin_sdf_points", "kin_program_dump", "kin_pose_residual", "kin_pose_residual_multi", "kin_probe_fp64",
           "kin_jit_status", "kin_jit_stats", "kin_codegen_dump", "kin_ik_solve", "kin_host_transfer_bytes",
           "kin_model_set_self_pairs", "kin_model_n_self_pairs", "kin_self_collision", "kin_ik_solve_self",
           "kin_ik_solve_links", "kin_grid_create", "kin_grid_set_values", "kin_grid_destroy", "kin_model_set_scene",
           "kin_sdf_points_scene"]


def source_files():
    """Every file the library is compiled from (the build id is their digest)."""
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cpp", ".cuh", ".h", ".hpp"))] + \
           [os.path.join(os.path.dirname(HERE), "include", "kin_b200.h")]


def source_id() -> str:
    """sha256 (first 16 hex digits) over the names and contents of csrc/* and include/kin_b200.h."""
    h = hashlib.sha256()
    for f in source_files():
        h.update(os.path.basename(f).encode() + b"\0")
        h.update(open(f, "rb").read())
        h.update(b"\0")
    return h.hexdigest()[:16]


def so_path(debug: bool = False) -> str:
    return SO_PATH_DEBUG if debug else SO_PATH


_ID_MARKER = b"KIN_BUILD_ID="


def so_build_id(path: str):
    """Build id of a built library, or None when it is missing / predates the build id.  Read from the file
    (the id is stored behind a marker string) rather than through dlopen, which would pin the old mapping."""
    if not os.path.exists(path):
        return None
    data = open(path, "rb").read()
    i = data.find(_ID_MARKER)
    if i < 0:
        return None
    j = data.find(b"\0", i)
    return data[i + len(_ID_MARKER):j].decode(errors="replace")


def needs_build(debug: bool = False) -> bool:
    return so_build_id(so_path(debug)) != source_id()


def _embed_object() -> str:
    """ld -r -b binary: the two header texts NVRTC needs at run time as one relocatable object
    (_binary_<file>_start / _end symbols; run inside csrc/ so that the names carry no directory)."""
    obj = os.path.join(HERE, "build", "kin_embedded.o")
    os.makedirs(os.path.dirname(obj), exist_ok=True)
    out = subprocess.run(["ld", "-r", "-b", "binary", "-z", "noexecstack", "-o", obj] + EMBEDDED, cwd=CSRC, capture_output=True, text=True)
    if out.returncode != 0:
        raise KinError("ld -b binary failed:\n" + out.stdout + out.stderr)
    return obj


def _nvcc_cmd(debug: bool, verbose: bool):
    return ["nvcc"] + NVCC_FLAGS + (["-DKIN_DEBUG"] if debug else []) + ['-DKIN_BUILD_ID="%s"' % source_id()] + \
           (["-Xptxas", "-v"] if verbose else []) + ["-o", so_path(debug)] + [os.path.join(CSRC, s) for s in SOURCES] + \
           [_embed_object(), "-ldl"]


def build(force: bool = False, verbose: bool = False, debug: bool = False, both: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> kinematics.jl_b200/libkin_b200.so (in-tree).
    ``debug=True`` builds libkin_b200_debug.so with -DKIN_DEBUG (bounds-checked table / scratch indices);
    ``both=True`` builds the two libraries side by side (two nvcc processes)."""
    variants = [False, True] if both else [debug]
    procs = []
    for dbg in variants:
        if force or needs_build(dbg):
            procs.append((dbg, subprocess.Popen(_nvcc_cmd(dbg, verbose), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    for dbg, pr in procs:
        out, err = pr.communicate()
        if pr.returncode != 0:
            raise KinError("nvcc failed (%s build):\n" % ("debug" if dbg else "release") + out + err)
        if verbose:
            print(err)
    return so_path(debug)


_LIB = None


def _find_nvrtc():
    """libnvrtc of the CUDA toolkit, else the one bundled with the torch wheels (nvidia/cuda_nvrtc)."""
    import glob
    pats = ["/usr/local/cuda/lib64/libnvrtc.so.1[0-9]", "/usr/local/cuda/targets/*/lib/libnvrtc.so.1[0-9]"]
    try:
        import nvidia
        for base in getattr(nvidia, "__path__", []):
            pats.append(os.path.join(base, "cuda_nvrtc", "lib", "libnvrtc.so.1[0-9]"))
    except ImportError:
        pass
    for p in pats:
        hits = sorted(glob.glob(p))
        if hits:
            return hits[-1]
    return None


def lib():
    """Load libkin_b200.so (libkin_b200_debug.so when KIN_DEBUG=1 is set); raises KinError when it has not been
    built or was built from other sources than the ones beside it (no fallback path exists)."""
    global _LIB
    if _LIB is None:
        debug = os.environ.get("KIN_DEBUG", "") not in ("", "0")
        path = so_path(debug)
        if not os.path.exists(path):
            raise KinError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'`; "
                           "there is no CPU fallback" % path)
        if "KIN_NVRTC_PATH" not in os.environ:          # where kin_jit.cpp should dlopen NVRTC from
            cand = _find_nvrtc()
            if cand:
                os.environ["KIN_NVRTC_PATH"] = cand
        L = C.CDLL(path)
        try:
            L.kin_build_id.restype = C.c_char_p
            built = L.kin_build_id().decode()
        except AttributeError:
            built = "none"
        if built != source_id() and not os.environ.get("KIN_ALLOW_STALE_SO"):
            raise KinError("%s was built from other sources (build id %s, sources on disk %s): rebuild with "
                           "`python -c 'import __graft_entry__ as g; g.build()'`" % (path, built, source_id()))
        L.kin_last_error.restype = C.c_char_p
        L.kin_abi_version.restype = C.c_int
        L.kin_debug_build.restype = C.c_int
        L.kin_model_create.argtypes = [C.POINTER(KinModelDesc), C.POINTER(C.c_void_p)]
        L.kin_model_destroy.argtypes = [C.c_void_p]
        L.kin_model_set_spheres.argtypes = [C.c_void_p, C.c_int32, _ip, _dp, _dp]
        L.kin_model_set_boxes.argtypes = [C.c_void_p, C.c_int32, _dp, _dp]
        L.kin_model_set_primitives.argtypes = [C.c_void_p, C.c_int32, _ip, _dp, _dp]
        L.kin_sdf_points_prims.argtypes = [C.c_int32, _ip, _dp, _dp, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_int32,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_model_set_scene.argtypes = [C.c_void_p, C.c_int32, _ip, _dp, _dp, C.POINTER(C.c_void_p)]
        L.kin_sdf_points_scene.argtypes = [C.c_int32, _ip, _dp, _dp, C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_void_p,
                                           C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_grid_create.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.POINTER(C.c_void_p)]
        L.kin_grid_set_values.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_grid_destroy.argtypes = [C.c_void_p]
        for f in (L.kin_model_n_dof, L.kin_model_n_spheres, L.kin_model_n_boxes):
            f.argtypes = [C.c_void_p]
        L.kin_eval.argtypes = [C.c_void_p, C.POINTER(KinCall)]
        L.kin_eval_host.argtypes = [C.c_void_p, C.POINTER(KinCall)]
        L.kin_launch_count.restype = C.c_int64
        L.kin_query_launch.argtypes = [C.c_void_p, C.POINTER(KinCall), _ip, _ip, _ip, _ip]
        L.kin_sdf_points.argtypes = [C.c_int32, _dp, _dp, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_int32,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_collision_summary.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_double, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_model_set_self_pairs.argtypes = [C.c_void_p, C.c_int32, _ip]
        L.kin_model_n_self_pairs.argtypes = [C.c_void_p]
        L.kin_self_collision.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_double, C.c_double,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_pose_residual.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                        C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_pose_residual_multi.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, _ip, _ip,
                                              C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_probe_fp64.argtypes = [_dp, _dp, _dp]
        L.kin_ik_solve.argtypes = [C.c_void_p, C.POINTER(KinIkCall)]
        L.kin_ik_solve_self.argtypes = [C.c_void_p, C.POINTER(KinIkCall), C.c_double, C.c_void_p]
        L.kin_ik_solve_links.argtypes = [C.c_void_p, C.POINTER(KinIkCall), C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                         C.c_int32, C.c_double, C.c_void_p]
        L.kin_jit_status.restype = C.c_char_p
        _lp = C.POINTER(C.c_int64)
        L.kin_jit_stats.argtypes = [_lp, _lp, _lp, _lp]
        L.kin_host_transfer_bytes.argtypes = [_lp, _lp, _lp]
        L.kin_codegen_dump.argtypes = [C.POINTER(KinModelDesc), C.POINTER(KinCall), C.c_int32, C.c_char_p]
        L.kin_program_dump.argtypes = [C.POINTER(KinModelDesc), _ip, C.c_int32, _ip, C.c_int32, C.c_int32, C.c_int32,
                                       _ip, C.c_int32, _ip, C.c_int32, _dp, C.c_int32]
        _LIB = L
    return _LIB


def check(rc: int):
    if rc != 0:
        raise KinError("libkin_b200 error %d: %s" % (rc, lib().kin_last_error().decode()))
