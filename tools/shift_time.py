#!/usr/bin/env python3
"""Staggered reads (--max-shift): kernel-only rate and the CLI's count_s.

(a) Kernel: 50 M x 75 bp device-resident reads (3.8 GB, larger than the L2) and the 77 441-guide
    Brunello-shaped library, Permuter on, offset 5.  Two samples: the synthetic sample with its guide at
    offset 5, and the same sample with 0-8 random bases put in front of every read (a staggered
    forward-primer mix, the guide at offset 5 + 0..8).  S = 1 is today's streaming kernel; S = 2, 4, 8
    the shift kernel.  One untimed submit first (it carries the skew plan), then CUDA events around
    five submits of the whole batch; the matched fraction is printed beside each rate.
(b) CLI: count_s of `sgcount` on one BGZF sample of 16.7 M reads with --max-shift 1 and --max-shift 8,
    five rounds, alternated.
usage: shift_time.py [n_reads [cli_reads]]"""
import json
import os
import statistics
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import sgcount_b200 as sg
from sgcount_b200 import synth

N = int(sys.argv[1]) if len(sys.argv) > 1 else 50_000_000
CLI_READS = int(sys.argv[2]) if len(sys.argv) > 2 else 1 << 24
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0xB2000002
L, STRIDE, OFFSET = 75, 76, 5

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True)
print(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi: {smi.stdout.strip().splitlines()[0] if smi.stdout else 'n/a'}",
      flush=True)

arr = synth.make_library(SEED, 77441, 20)
library = sg.Library([arr[i].tobytes() for i in range(len(arr))], [b"g%d" % i for i in range(len(arr))])
permuter = sg.Permuter.new(library)
sample = synth.Sample(SEED, 0, arr, L, OFFSET, False)
d = torch.empty(N * STRIDE + 256, dtype=torch.uint8, device="cuda")
sample.fill_device(0, N, d.data_ptr())
torch.cuda.synchronize()


def stagger(buf):
    """0..8 random A/C/G/T bases in front of every read, the read's end cut off to keep 75 bp"""
    rows = buf[:N * STRIDE].view(N, STRIDE)
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(SEED)
    shift = torch.randint(0, 9, (N,), device="cuda", generator=gen)
    for s in range(1, 9):
        idx = (shift == s).nonzero().squeeze(1)
        sub = rows[idx]
        prefix = acgt[torch.randint(0, 4, (len(idx), s), device="cuda", generator=gen)]
        rows[idx] = torch.cat([prefix, sub[:, :L - s], sub[:, L:]], dim=1)
        del idx, sub, prefix
    torch.cuda.synchronize()


def kernel_rate(S):
    c = sg.Counter(library, permuter, sg.Offset.Forward(OFFSET), max_shift=S)
    c.submit_device(d.data_ptr(), N * STRIDE, N, STRIDE, L)  # the skew plan, warm-up
    torch.cuda.synchronize()
    c.reset()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        c.submit_device(d.data_ptr(), N * STRIDE, N, STRIDE, L)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 5
    _, total, matched = c.finish()
    return ms, matched / total, c.launch_info().kernel


for label in ("offset 5, no stagger", "offset 5 + 0..8 stagger"):
    if "stagger" in label and "no" not in label:
        stagger(d)
    for S in (1, 2, 4, 8):
        ms, frac, kernel = kernel_rate(S)
        print(f"{label:<26} S={S:<2} kernel={kernel}: {ms:8.3f} ms per {N} reads  {N / ms / 1e6:6.3f} G reads/s  "
              f"matched {frac:.4f}", flush=True)
del d
torch.cuda.empty_cache()

tmp = tempfile.mkdtemp(prefix="sgc_shift_")
lib = os.path.join(tmp, "lib.fa")
with open(lib, "wb") as f:
    f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
path = os.path.join(tmp, "s.fastq.gz")
synth.Sample(SEED, 1, arr, L, 9, False).write_fastq_bgzf(path, 0, CLI_READS, gz_level=1)
print(f"CLI sample: {CLI_READS} reads, {os.path.getsize(path) / 1e6:.0f} MB of BGZF", flush=True)
times = {1: [], 8: []}
for rnd in range(5):
    for S in ((1, 8) if rnd % 2 == 0 else (8, 1)):
        p = subprocess.run([EXE, "-l", lib, "-i", path, "-o", os.path.join(tmp, f"t{S}.tsv"), "--timing", "--max-shift", str(S)],
                           capture_output=True, text=True)
        assert p.returncode == 0, p.stderr
        t = json.loads([l for l in p.stderr.splitlines() if l.startswith("{")][-1])
        fin = [l for l in p.stderr.splitlines() if l.startswith("Finished:")][0]
        assert t["device_ingest_samples"] == 1 and t["max_shift"] == S, t
        times[S].append(t["count_s"])
        print(f"round {rnd} --max-shift {S}: count_s {t['count_s']:.3f}  {t['reads'] / t['count_s'] / 1e9:.3f} G reads/s  "
              f"{fin.split(';', 1)[1].strip()}", flush=True)
for S, ts in times.items():
    print(f"--max-shift {S}: count_s best {min(ts):.3f} / median {statistics.median(ts):.3f} s over {len(ts)} runs", flush=True)
