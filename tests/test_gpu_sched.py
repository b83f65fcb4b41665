"""GPU: the claimed-tile schedule of the FK / Jacobian-only specialised kernels (kin_gen_skeleton.cuh, KSCHED: tiles
claimed from a counter, inputs prefetched into L2 one epoch at a time).  Every case runs three ways on the same inputs:
the interpreting kernel (KIN_DISABLE_JIT), the specialised kernel with static tiles (KIN_JIT_SCHED_MIN_N above n: the
schedule -- and the constant-row fill -- off) and with claimed tiles.  Static against claimed tiles, the whole output
storage must be equal bit for bit (padding and the words in front of an offset pointer hold a sentinel nobody may
overwrite); against the interpreting kernel the values must be equal (== : the sign of a folded zero is the one thing
specialisation changes).  AoS calls run the input batches there instead (kin_b200.cu: gen_options), checked the same
way.  Small epochs (KIN_JIT_EPOCH_MB=1: 128 tiles of 128 configurations in FP64) put the epoch
boundaries where the cases want them."""
import ctypes as C

import numpy as np
import pytest
import torch

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import device_model
import scenes

pytestmark = pytest.mark.gpu

SENTINEL = -12345.0
EPOCH = 128 * 128           # configurations per epoch at KIN_JIT_EPOCH_MB=1 (FP64, 8 columns, 128 threads)
BIG = (1 << 18) + 77        # at and above kSchedMinBatch (kin_b200.cu), ragged
KNOBS = ("KIN_DISABLE_JIT", "KIN_FORCE_JIT", "KIN_JIT_SCHED_MIN_N", "KIN_JIT_EPOCH_MB")


def _setup(layout, q, n, pad, off, dt, fk, jac):
    """Inputs and sentinel-filled outputs of one call in `layout`; returns (KinCall, outputs, keep-alive)."""
    nd = q.shape[1]
    qt = torch.as_tensor(q, device="cuda").to(dt)                                  # [n][nd]
    n32 = (n + 31) // 32 * 32
    if layout == "soa":
        ld = n + pad
        Q = torch.zeros((nd, ld), dtype=dt, device="cuda")
        Q[:, :n] = qt.t()
    elif layout == "tiled":
        ld = 0
        Q = torch.zeros((n32, nd), dtype=dt, device="cuda")
        Q[:n] = qt
        Q = Q.view(n32 // 32, 32, nd).permute(0, 2, 1).contiguous()
    else:
        ld, Q = 0, qt.contiguous()
    cols = ld if layout == "soa" else (n32 if layout == "tiled" else n)
    ip = C.POINTER(C.c_int32)
    c = L.KinCall()
    c.precision = L.F32 if dt == torch.float32 else L.F64
    c.layout = {"soa": L.SOA, "tiled": L.TILED32, "aos": L.AOS}[layout]
    c.n, c.batch_stride, c.q = n, ld, Q.data_ptr()
    es = torch.empty((), dtype=dt).element_size()
    out = {}
    if fk is not None:
        T = torch.full((off + 12 * len(fk) * cols,), SENTINEL, dtype=dt, device="cuda")
        c.n_fk_links, c.fk_links, c.T_out = len(fk), fk.ctypes.data_as(ip), T.data_ptr() + off * es
        out["T"] = T
    if jac is not None:
        J = torch.full((off + 6 * nd * len(jac) * cols,), SENTINEL, dtype=dt, device="cuda")
        c.n_jac_links, c.jac_links, c.J_out, c.with_rot = len(jac), jac.ctypes.data_as(ip), J.data_ptr() + off * es, 1
        out["J"] = J
    c.truncation_dist = float("inf")
    return c, out, (Q, fk, jac)


def _env(monkeypatch, env):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _bits(t):
    return t.view(torch.int64 if t.dtype == torch.float64 else torch.int32)


def _model():
    m, joints, _ = scenes.product_fetch(False)
    _, jo, _ = scenes.oracle_fetch(False)
    K.set_joint_angles(m, joints, torch.zeros((1, len(joints)), dtype=torch.float64, device="cuda"))
    return m, jo, device_model(m), L.lib()


def _calls(m, outs):
    fk = np.arange(1, 26, dtype=np.int32) if "T" in outs else None
    # a J-only call of the gripper alone writes too little per configuration for the schedule: all links then
    jac = np.array([K.find_link(m, "gripper_link").id] if "T" in outs else list(range(1, 26)), dtype=np.int32) if "J" in outs else None
    return fk, jac


@pytest.mark.parametrize("layout, n, pad, off, prec, outs, epoch_mb", [
    ("soa", EPOCH - 5, 0, 0, "f64", "TJ", 1),       # less than one epoch
    ("soa", EPOCH, 0, 0, "f64", "TJ", 1),           # exactly one epoch
    ("soa", EPOCH - 128, 0, 0, "f64", "TJ", 1),     # one epoch - 1 tile
    ("soa", EPOCH + 128, 0, 0, "f64", "TJ", 1),     # one epoch + 1 tile
    ("soa", 5 * EPOCH + 77, 3, 1, "f64", "TJ", 1),  # several epochs, ragged, batch_stride % 4 != 0, offset pointers
    ("soa", BIG, 0, 0, "f64", "TJ", None),          # the default epochs
    ("soa", BIG, 64, 0, "f64", "TJ", None),         # padded batch_stride
    ("soa", BIG, 3, 1, "f32", "TJ", None),
    ("soa", BIG, 3, 1, "f64", "T", None),
    ("soa", BIG, 3, 1, "f64", "J", None),
    ("tiled", BIG, 0, 0, "f64", "TJ", None),
    ("tiled", EPOCH + 128 + 5, 0, 0, "f64", "TJ", 1),
    ("tiled", BIG, 0, 0, "f32", "TJ", None),
    ("aos", BIG, 0, 0, "f64", "TJ", None),
    ("aos", EPOCH - 5, 0, 0, "f64", "TJ", 1),
    ("aos", BIG, 0, 0, "f64", "J", None),
])
def test_claimed_tiles_match_static_tiles_bitwise(layout, n, pad, off, prec, outs, epoch_mb, monkeypatch):
    m, jo, dm, lib = _model()
    q = scenes.random_configs(jo, n, False, seed=43)
    dt = torch.float32 if prec == "f32" else torch.float64
    fk, jac = _calls(m, outs)
    res = {}
    sched = {"KIN_FORCE_JIT": "1", "KIN_JIT_SCHED_MIN_N": "0"}
    if epoch_mb:
        sched["KIN_JIT_EPOCH_MB"] = str(epoch_mb)
    for name, env in (("interp", {"KIN_DISABLE_JIT": "1"}), ("static", {"KIN_FORCE_JIT": "1", "KIN_JIT_SCHED_MIN_N": str(1 << 40)}),
                      ("sched", sched)):
        _env(monkeypatch, env)
        c, out, keep = _setup(layout, q, n, pad, off, dt, fk, jac)
        c.stream = torch.cuda.current_stream().cuda_stream
        L.check(lib.kin_eval(dm.h, C.byref(c)))
        torch.cuda.synchronize()
        res[name] = out
    for key in res["interp"]:
        a, b, r = res["sched"][key], res["static"][key], res["interp"][key]
        assert torch.equal(_bits(a), _bits(b)), key
        if layout == "tiled":
            # the last tile's slots past n: the TMA stores of the specialised kernels write whole 32-configuration
            # blocks (the last configuration again), the interpreting kernel leaves them alone
            n32 = (n + 31) // 32 * 32
            valid = (torch.arange(n32, device=a.device).view(n32 // 32, 1, 32) < n).expand(n32 // 32, a.numel() // n32, 32)
            assert torch.equal(a[valid.reshape(-1)], r[valid.reshape(-1)]), key
        else:
            assert torch.equal(a, r), key
        assert bool((a[:off] == SENTINEL).all()), key
        if layout == "soa":
            rows = a[off:].view(-1, n + pad)
            assert bool((rows[:, n:] == SENTINEL).all()) and not bool((rows[:, :n] == SENTINEL).any()), key
        elif layout == "aos":
            assert not bool((a == SENTINEL).any()), key
    compiles, hits, launches, failures = (C.c_int64() for _ in range(4))
    lib.kin_jit_stats(C.byref(compiles), C.byref(hits), C.byref(launches), C.byref(failures))
    assert failures.value == 0 and launches.value > 0


def test_concurrent_launches_on_two_streams_keep_their_own_counters(monkeypatch):
    """Two claimed-tile calls in flight at once on two streams (each launch takes its own zeroed counter from the
    stream-ordered pool): both equal, bit for bit, what each computes alone."""
    m, jo, dm, lib = _model()
    fk, jac = _calls(m, "TJ")
    _env(monkeypatch, {"KIN_FORCE_JIT": "1", "KIN_JIT_SCHED_MIN_N": "0", "KIN_JIT_EPOCH_MB": "1"})
    qs = [scenes.random_configs(jo, n, False, seed=s) for n, s in ((3 * EPOCH + 77, 51), (2 * EPOCH + 5, 52))]
    alone, keep = [], []
    for q in qs:
        c, out, k = _setup("soa", q, len(q), 0, 0, torch.float64, fk, jac)
        c.stream = torch.cuda.current_stream().cuda_stream
        L.check(lib.kin_eval(dm.h, C.byref(c)))
        torch.cuda.synchronize()
        alone.append(out)
        keep.append(k)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    together = []
    for rep in range(3):
        calls = []
        for q, s in zip(qs, streams):
            c, out, k = _setup("soa", q, len(q), 0, 0, torch.float64, fk, jac)
            torch.cuda.synchronize()
            c.stream = s.cuda_stream
            calls.append((c, out, k))
        for c, _, _ in calls:
            L.check(lib.kin_eval(dm.h, C.byref(c)))
        torch.cuda.synchronize()
        together.append([o for _, o, _ in calls])
    for outs in together:
        for a, b in zip(outs, alone):
            for key in b:
                assert torch.equal(_bits(a[key]), _bits(b[key])), key
