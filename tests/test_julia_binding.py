"""The Julia binding (julia/CUDABackend.jl) cannot be executed here (no julia).  What can be checked without it:
its two struct declarations against the C structs as gcc lays them out (tests/abi_layout.c), the ctypes structures of
the Python mirror against the same dump, every `ccall` against the declarations of include/kin_b200.h (symbol exists,
argument count and argument classes match), and that every name it imports from the reference exists there."""
import ctypes as C
import json
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
JL = open(os.path.join(ROOT, "julia", "CUDABackend.jl")).read()
HDR = open(os.path.join(ROOT, "include", "kin_b200.h")).read()

# Julia type -> (size, alignment, class) under the C ABI Julia uses for isbits structs
JL_TYPES = {"Cint": (4, 4, "i32"), "Int64": (8, 8, "i64"), "Cdouble": (8, 8, "f64")}


def jl_type(t):
    t = t.strip()
    if t.startswith(("Ptr{", "CuPtr{", "Ref{")) or t == "Cstring":
        return 8, 8, "ptr"
    return JL_TYPES[t]


@pytest.fixture(scope="module")
def c_layout(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("abi") / "abi_layout")
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(ROOT, "tests", "abi_layout.c")])
    return json.loads(subprocess.check_output([exe]))


def julia_struct(name):
    body = re.search(r"^struct %s\n(.*?)^end" % name, JL, re.S | re.M).group(1)
    return [tuple(x.strip() for x in line.split("::")) for line in body.strip().splitlines()]


@pytest.mark.parametrize("name", ["KinModelDesc", "KinCall", "KinIkCall"])
def test_julia_struct_matches_c_layout(name, c_layout):
    fields = julia_struct(name)
    ref = c_layout[name]["fields"]
    assert [f[0] for f in fields] == [r["name"] for r in ref]           # same fields, same order
    off, max_al = 0, 1
    for (fname, ftype), r in zip(fields, ref):
        size, al, _ = jl_type(ftype)
        off = (off + al - 1) // al * al
        assert (off, size) == (r["offset"], r["size"]), (fname, ftype, off, size, r)
        off += size
        max_al = max(max_al, al)
    assert (off + max_al - 1) // max_al * max_al == c_layout[name]["size"]


@pytest.mark.parametrize("name", ["KinModelDesc", "KinCall", "KinIkCall"])
def test_ctypes_struct_matches_c_layout(name, c_layout):
    from kinematics_jl_b200 import lib as L
    S = getattr(L, name)
    ref = c_layout[name]["fields"]
    assert [f[0] for f in S._fields_] == [r["name"] for r in ref]
    for (fname, _), r in zip(S._fields_, ref):
        d = getattr(S, fname)
        assert (d.offset, d.size) == (r["offset"], r["size"]), fname
    assert C.sizeof(S) == c_layout[name]["size"]


def c_declarations():
    """name -> list of argument classes, from the KIN_API declarations of the header."""
    out = {}
    for m in re.finditer(r"KIN_API\s+([^;(]*?)\b(kin_\w+)\s*\(([^;]*?)\)\s*;", HDR, re.S):
        args = [a.strip() for a in m.group(3).replace("\n", " ").split(",")]
        classes = []
        for a in args:
            if a == "void":
                continue
            if "*" in a:
                classes.append("ptr")
            elif a.startswith("double"):
                classes.append("f64")
            elif a.startswith("int64_t"):
                classes.append("i64")
            elif a.startswith(("int32_t", "int")):
                classes.append("i32")
            else:
                raise AssertionError("unclassified C parameter: " + a)
        out[m.group(2)] = classes
    return out


def test_every_ccall_matches_the_header():
    decl = c_declarations()
    calls = re.findall(r"ccall\(\(:(\w+), libkin\),\s*(\w+),\s*\(([^()]*)\)", JL)
    assert len(calls) >= 8
    seen = set()
    for sym, ret, argt in calls:
        assert sym in decl, "ccall of a symbol the header does not declare: " + sym
        seen.add(sym)
        types = [t for t in (x.strip() for x in argt.split(",")) if t]
        got = [jl_type(t)[2] for t in types]
        assert got == decl[sym], (sym, got, decl[sym])
        assert ret in ("Cint", "Cstring")
    # the operators of the reference's export list (Kinematics.jl:45-70) on this path all have a binding
    assert {"kin_model_create", "kin_model_destroy", "kin_model_set_boxes", "kin_eval", "kin_eval_host", "kin_pose_residual_multi",
            "kin_sdf_points", "kin_last_error", "kin_ik_solve"} <= seen
    for fn in ("get_transform", "get_jacobian", "get_jacobian!", "compute_coll_dists", "compute_coll_dists_and_grads", "ineq_const",
               "f_objective", "pose_constraint", "sdf_points", "sdf_gradient", "eval_host!", "set_boxes!", "inverse_kinematics_batch"):
        assert re.search(r"^(function )?%s\(" % re.escape(fn), JL, re.M), fn


def test_imported_reference_names_exist():
    """Every name the module imports from Kinematics is defined in the reference's src/ -- an unbound name was the
    round-1 bug (Kinematics.inv_pose).  The Julia sources of Kinematics.jl are not part of this repository: that part
    runs where KIN_REFERENCE_SRC names the reference's src/ directory, and skips elsewhere."""
    names = set()
    for m in re.finditer(r"^(?:using|import) \.\.Kinematics: (.*?)(?=^\S|\Z)", JL, re.S | re.M):
        names |= {n.strip() for n in m.group(1).replace("\n", " ").split(",") if n.strip()}
    assert {"inv_pose", "get_jacobian!", "Mechanism", "translation", "rpy"} <= names
    assert "Kinematics." not in re.sub(r"\.\.Kinematics", "", JL.split("module CUDABackend")[1])   # no unqualified module access
    src = os.environ.get("KIN_REFERENCE_SRC", "")
    if not os.path.isdir(src):
        pytest.skip("the reference's Julia sources are not present (set KIN_REFERENCE_SRC to its src/ directory)")
    text = "\n".join(open(os.path.join(src, f)).read() for f in os.listdir(src) if f.endswith(".jl"))
    for n in names:
        e = re.escape(n)
        pat = r"(function\s+%s(?![\w!])|(?<![\w.])%s\([^)\n]*\)\s*(where [^=\n]*)?=|struct\s+%s\b|abstract type %s\b|^\s*%s\s*=|const %s\b)" % ((e,) * 6)
        assert re.search(pat, text, re.M) or n in ("Fixed", "Revolute", "Prismatic"), n
