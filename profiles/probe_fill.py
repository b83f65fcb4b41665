"""Probe: the write ceiling of this B200 next to the headline's output pattern (DESIGN 4.4).

Runs, in one process tree on one GPU: the card's name / power limit / max SM clock (nvidia-smi, read-only), torch.fill_
of 8 GiB (the 7.5 TB/s figure of probe_write_bw.py), then `probe_store fill` (contiguous 8 GiB fills with each store
form, and the 348-row SoA pattern at 2^22 configurations with its 175 constant rows as contiguous fills), then torch.fill_
again.  `python profiles/probe_fill.py sched [rounds]` instead runs `probe_store sched`: the 173 varying rows under the
static / barrier schedule against claimed tiles with and without epoch L2 prefetches, and short-lived CTAs (DESIGN 4.4).
Usage: python profiles/probe_fill.py [sched] [rounds]"""
import os
import shutil
import subprocess
import sys
import tempfile

import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def torch_fill(rounds):
    x = torch.empty(1 << 30, dtype=torch.float64, device="cuda")       # 8 GiB
    for _ in range(3):
        x.fill_(1.0)
    torch.cuda.synchronize()
    ms = []
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            x.fill_(1.0)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b) / 5)
    del x
    torch.cuda.empty_cache()
    ms.sort()
    med = ms[len(ms) // 2]
    print("%-48s %9.4f %9.4f %9.4f %9.1f" % ("torch.fill_ 8 GiB", med, ms[0], ms[-1], 8 * (1 << 30) / (med * 1e-3) / 1e9), flush=True)


def main():
    args = sys.argv[1:]
    sched = bool(args) and args[0] == "sched"
    if sched:
        args = args[1:]
    rounds = int(args[0]) if args else 7
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout, flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "probe_store")
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        subprocess.check_call([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                               os.path.join(HERE, "probe_store.cu")])
        if sched:
            subprocess.check_call([exe, "sched", str(rounds)])
            return
        torch_fill(rounds)
        subprocess.check_call([exe, "fill", str(rounds)])
        torch_fill(rounds)


if __name__ == "__main__":
    main()
