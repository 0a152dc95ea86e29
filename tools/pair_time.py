#!/usr/bin/env python3
"""Dual-guide constructs (sgc_pair_counter): kernel-only rate of paired counting.

50 M pairs x 2 x 75 bp device-resident reads (7.6 GB, larger than the L2), offset 5, Permuter on, synthetic
bench mix (sgcount_b200.synth) in both mates; both mates are drawn with the same seed so that read i of
mate 2 carries the guide of the same index as read i of mate 1.
  - all-by-all: two libraries of 300 guides, 90 000 constructs;
  - 1:1: two libraries of 77 441 guides, construct j = (j, j).
For each: one untimed submit (it carries the skew plans), then CUDA events around five submits of the whole
batch (the report on, capacity 2^22); beside it, one mate counted alone by an ordinary counter (the
streaming kernel), and the tallies of the last run.
usage: pair_time.py [n_pairs]"""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import sgcount_b200 as sg
from sgcount_b200 import synth

N = int(sys.argv[1]) if len(sys.argv) > 1 else 50_000_000
SEED = 0xB2000012
L, STRIDE, OFFSET = 75, 76, 5
CAPACITY = 1 << 22
RUNS = 5

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True)
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi: {smi.stdout.strip().splitlines()[0] if smi.stdout else 'n/a'}",
      flush=True)


def timed(fn):
    ms = []
    for _ in range(RUNS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return min(ms), statistics.median(ms)


def case(name, n_guides, pairs):
    arrs = [synth.make_library(SEED + m, n_guides, 20) for m in (0, 1)]
    libs = [sg.Library([a[i].tobytes() for i in range(len(a))], [b"g%d" % i for i in range(len(a))]) for a in arrs]
    perms = [sg.Permuter.new(lib) for lib in libs]
    bufs = []
    for m in (0, 1):
        d = torch.empty(N * STRIDE + 256, dtype=torch.uint8, device="cuda")
        synth.Sample(SEED, 0, arrs[m], L, OFFSET, False).fill_device(0, N, d.data_ptr())
        bufs.append(d)
    torch.cuda.synchronize()
    off = sg.Offset.Forward(OFFSET)
    c1, c2 = sg.Counter(libs[0], perms[0], off), sg.Counter(libs[1], perms[1], off)
    pc = sg.PairCounter(c1, c2, pairs, CAPACITY)

    def submit():
        pc.submit_device(N, bufs[0].data_ptr(), N * STRIDE, bufs[1].data_ptr(), N * STRIDE, stride1=STRIDE, read_len1=L,
                         stride2=STRIDE, read_len2=L)

    submit()
    pc.reset()
    best, med = timed(submit)
    _, info = pc.finish()
    single = sg.Counter(libs[0], perms[0], off)
    single.submit_device(bufs[0].data_ptr(), N * STRIDE, N, STRIDE, L)
    s_best, s_med = timed(lambda: single.submit_device(bufs[0].data_ptr(), N * STRIDE, N, STRIDE, L))
    per = {k: info[k] / info["total"] for k in ("listed", "recombined", "first_only", "second_only", "neither")}
    print(f"{name}: {len(pairs)} constructs, {N} pairs: paired {best:.3f} / {med:.3f} ms best / median = "
          f"{N / best / 1e6:.2f} G pairs/s; one mate alone (streaming kernel) {s_best:.3f} / {s_med:.3f} ms = "
          f"{N / s_best / 1e6:.2f} G reads/s; last run of {RUNS}: "
          + ", ".join(f"{k} {v:.3f}" for k, v in per.items()) + f", report distinct {info['distinct']}, overflow "
          f"{info['overflow']}", flush=True)
    del pc


case("all-by-all 300 x 300", 300, [(i, j) for i in range(300) for j in range(300)])
case("1:1 77 441", 77441, [(j, j) for j in range(77441)])
