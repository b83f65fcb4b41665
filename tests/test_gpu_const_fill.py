"""GPU: the configuration-independent rows of the SoA FK / Jacobian outputs of the input-batched specialised kernel,
written as contiguous fills by kin_const_fill_kernel (kin_gen_skeleton.cuh).  Every case runs three ways on the same
inputs: the interpreting kernel (KIN_DISABLE_JIT), the specialised kernel without the fill (KIN_JIT_CONST_FILL=0: every
row stored per thread) and with it (the default).  With and without the fill the whole output storage must be equal bit
for bit -- padding columns and the words in front of an offset pointer included, which hold a sentinel nobody may
overwrite; against the interpreting kernel the values must be equal (== : the sign of a folded zero is the one thing
specialisation changes)."""
import ctypes as C

import numpy as np
import pytest
import torch

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import device_model
import scenes

pytestmark = pytest.mark.gpu

QB_MIN = 1 << 18           # kin_b200.cu: kQbatchMinBatch, the smallest batch that gets input batching (and the fill)
SENTINEL = -12345.0


def _run(dm, lib, q, n, ld, off, dt, fk, jac, env, monkeypatch):
    """One kin_eval with SoA q / T / J of leading dimension ld, T / J pointers `off` elements into their storage."""
    for k in ("KIN_DISABLE_JIT", "KIN_FORCE_JIT", "KIN_JIT_CONST_FILL"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    nd = q.shape[1]
    Q = torch.zeros((nd, ld), dtype=dt, device="cuda")
    Q[:, :n] = torch.as_tensor(np.ascontiguousarray(q.T), device="cuda").to(dt)
    ip = C.POINTER(C.c_int32)
    c = L.KinCall()
    c.precision, c.layout, c.n, c.batch_stride, c.q = (L.F32 if dt == torch.float32 else L.F64), L.SOA, n, ld, Q.data_ptr()
    es = torch.empty((), dtype=dt).element_size()
    out = {}
    if fk is not None:
        T = torch.full((off + 12 * len(fk) * ld,), SENTINEL, dtype=dt, device="cuda")
        c.n_fk_links, c.fk_links, c.T_out = len(fk), fk.ctypes.data_as(ip), T.data_ptr() + off * es
        out["T"] = T
    if jac is not None:
        J = torch.full((off + 6 * nd * len(jac) * ld,), SENTINEL, dtype=dt, device="cuda")
        c.n_jac_links, c.jac_links, c.J_out, c.with_rot = len(jac), jac.ctypes.data_as(ip), J.data_ptr() + off * es, 1
        out["J"] = J
    c.truncation_dist = float("inf")
    c.stream = torch.cuda.current_stream().cuda_stream
    n0 = lib.kin_launch_count()
    L.check(lib.kin_eval(dm.h, C.byref(c)))
    torch.cuda.synchronize()
    out["launches"] = lib.kin_launch_count() - n0
    return out


def _bits(t):
    return t.view(torch.int64 if t.dtype == torch.float64 else torch.int32)


@pytest.mark.parametrize("n, pad, off, prec, outs", [
    (QB_MIN - 1, 0, 0, "f64", "TJ"),            # below the input-batching threshold: no fill
    (QB_MIN, 0, 0, "f64", "TJ"),
    (QB_MIN + 77, 0, 0, "f64", "TJ"),           # ragged n
    (QB_MIN, 64, 0, "f64", "TJ"),               # batch_stride > n, rows still 32-byte aligned
    (QB_MIN + 77, 3, 0, "f64", "TJ"),           # batch_stride % 4 != 0: every row starts on a different alignment
    (QB_MIN + 77, 5, 1, "f64", "TJ"),           # T / J pointers 8 bytes into their storage
    (QB_MIN + 77, 3, 1, "f32", "TJ"),
    (QB_MIN + 77, 3, 1, "f64", "T"),
    (QB_MIN + 77, 3, 1, "f64", "J"),
])
def test_constant_rows_filled_by_the_kernel_are_bitwise_the_stored_ones(n, pad, off, prec, outs, monkeypatch):
    m, joints, _ = scenes.product_fetch(False)
    _, jo, _ = scenes.oracle_fetch(False)
    K.set_joint_angles(m, joints, torch.zeros((1, len(joints)), dtype=torch.float64, device="cuda"))
    dm = device_model(m)
    lib = L.lib()
    # (no exact-zero angles: there the sign of a zero may differ between two compilations of phase 1)
    q = scenes.random_configs(jo, n, False, seed=41)
    dt = torch.float32 if prec == "f32" else torch.float64
    fk = np.arange(1, 26, dtype=np.int32) if "T" in outs else None
    # a J-only call of the gripper alone writes too little per configuration to be input-batched: all links then
    jac = np.array([K.find_link(m, "gripper_link").id] if "T" in outs else list(range(1, 26)), dtype=np.int32) if "J" in outs else None
    ld = n + pad
    args = (dm, lib, q, n, ld, off, dt, fk, jac)
    ref = _run(*args, {"KIN_DISABLE_JIT": "1"}, monkeypatch)
    stored = _run(*args, {"KIN_FORCE_JIT": "1", "KIN_JIT_CONST_FILL": "0"}, monkeypatch)
    filled = _run(*args, {"KIN_FORCE_JIT": "1"}, monkeypatch)
    assert stored["launches"] == 1 and filled["launches"] == (2 if n >= QB_MIN else 1)
    for key in ("T", "J"):
        if key not in ref:
            continue
        assert torch.equal(_bits(filled[key]), _bits(stored[key])), key
        assert torch.equal(filled[key], ref[key]), key
        rows = filled[key][off:].view(-1, ld)
        assert bool((filled[key][:off] == SENTINEL).all()) and bool((rows[:, n:] == SENTINEL).all()), key
        assert not bool((rows[:, :n] == SENTINEL).any()), key
    compiles, hits, launches, failures = (C.c_int64() for _ in range(4))
    lib.kin_jit_stats(C.byref(compiles), C.byref(hits), C.byref(launches), C.byref(failures))
    assert failures.value == 0 and launches.value > 0
