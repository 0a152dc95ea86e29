#!/usr/bin/env python3
"""Unmatched report (--unmatched-report): its kernel-only cost, the CLI's count_s with and without it, and
the host time to merge and write the report.

(a) Kernel: 50 M x 75 bp device-resident reads (3.8 GB, larger than the L2) and the 77 441-guide
    Brunello-shaped library, Permuter on, offset 5.  Report off (the streaming kernel) against report on
    (the line kernel, then unmatched_collect_kernel, capacity 2^22), on the synthetic bench mix and on the
    same reads with 30 % of them replaced by one adapter-dimer read and 10 % by random bases.  One untimed
    submit first (it carries the skew plan), then CUDA events around five submits of the whole batch.
(b) CLI: count_s of `sgcount` on a BGZF and a single-member gzip sample of 16.7 M reads, with and without
    --unmatched-report, five rounds alternated; the count tables must be identical.
(c) Host: unmatched_s of the CLI (compaction, copy, merge by window and the TSV) on plain FASTQ samples
    whose unmatched reads hold 10^5 and 4 * 10^6 distinct windows.
usage: unmatched_time.py [n_reads [cli_reads]]"""
import json
import os
import statistics
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import sgcount_b200 as sg
from sgcount_b200 import synth

N = int(sys.argv[1]) if len(sys.argv) > 1 else 50_000_000
CLI_READS = int(sys.argv[2]) if len(sys.argv) > 2 else 1 << 24
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0xB2000011
L, STRIDE, OFFSET = 75, 76, 5
CAPACITY = 1 << 22

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


def dimer_mix(buf):
    """30 % of the reads one adapter-dimer read, 10 % random A/C/G/T"""
    rows = buf[:N * STRIDE].view(N, STRIDE)
    gen = torch.Generator(device="cuda").manual_seed(SEED)
    acgt = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    u = torch.rand(N, device="cuda", generator=gen)
    dimer = acgt[torch.randint(0, 4, (L,), device="cuda", generator=gen)]
    idx = (u < 0.3).nonzero().squeeze(1)
    rows[idx, :L] = dimer
    idx = ((u >= 0.3) & (u < 0.4)).nonzero().squeeze(1)
    rows[idx, :L] = acgt[torch.randint(0, 4, (len(idx), L), device="cuda", generator=gen)]
    del idx, u
    torch.cuda.synchronize()


def kernel_rate(capacity):
    c = sg.Counter(library, permuter, sg.Offset.Forward(OFFSET), unmatched_capacity=capacity)
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
    counts, total, matched = c.finish()
    info = c.unmatched(3) if capacity else None
    return ms, counts, total, matched, c.launch_info(), info


for label in ("bench mix", "30 % dimer + 10 % junk"):
    if "dimer" in label:
        dimer_mix(d)
    res = {}
    for capacity in (None, CAPACITY):
        ms, counts, total, matched, li, info = kernel_rate(capacity)
        res[capacity] = (counts, total, matched)
        extra = f"  report: top {[(w.decode(), n) for w, n in info[0]]} {info[1]}" if info else ""
        print(f"{label:<24} report={'on ' if capacity else 'off'} kernel={li.kernel} replicas={li.replicas} hot={li.hot_guides}: "
              f"{ms:8.3f} ms per {N} reads  {N / ms / 1e6:6.3f} G reads/s  matched {matched / total:.4f}{extra}", flush=True)
    assert np.array_equal(res[None][0], res[CAPACITY][0]) and res[None][1:] == res[CAPACITY][1:], label
del d
torch.cuda.empty_cache()

tmp = tempfile.mkdtemp(prefix="sgc_unmatched_")
lib = os.path.join(tmp, "lib.fa")
with open(lib, "wb") as f:
    f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
paths = {"bgzf": os.path.join(tmp, "b.fastq.gz"), "gzip": os.path.join(tmp, "m.fastq.gz")}
synth.Sample(SEED, 1, arr, L, 9, False).write_fastq_bgzf(paths["bgzf"], 0, CLI_READS, gz_level=1)
synth.Sample(SEED, 1, arr, L, 9, False).write_fastq(paths["gzip"], 0, CLI_READS, reads_per_member=CLI_READS, gz_level=1)


def cli(path, report, tag):
    out = os.path.join(tmp, f"{tag}.tsv")
    args = [EXE, "-l", lib, "-i", path, "-a", "9", "-o", out, "--timing"]
    if report:
        args += ["--unmatched-report", os.path.join(tmp, f"{tag}.unmatched.tsv")]
    p = subprocess.run(args, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    t = json.loads([l for l in p.stderr.splitlines() if l.startswith("{")][-1])
    assert t["device_ingest_samples"] == 1 and (("unmatched_s" in t) == report), t
    with open(out, "rb") as f:
        return t, f.read()


for kind, path in paths.items():
    print(f"CLI sample ({kind}): {CLI_READS} reads, {os.path.getsize(path) / 1e6:.0f} MB", flush=True)
    times, tables = {False: [], True: []}, set()
    for rnd in range(5):
        for report in ((False, True) if rnd % 2 == 0 else (True, False)):
            t, table = cli(path, report, f"{kind}{int(report)}")
            tables.add(table)
            times[report].append(t["count_s"])
            print(f"round {rnd} {kind} report={'on ' if report else 'off'}: count_s {t['count_s']:.3f}  "
                  f"{t['reads'] / t['count_s'] / 1e9:.3f} G reads/s" + (f"  unmatched_s {t['unmatched_s']:.4f}" if report else ""),
                  flush=True)
    assert len(tables) == 1, "count tables differ"
    for report, ts in times.items():
        print(f"{kind} report={'on ' if report else 'off'}: count_s best {min(ts):.3f} / median {statistics.median(ts):.3f} s "
              f"over {len(ts)} runs; tables identical", flush=True)

rng = np.random.default_rng(SEED)
for distinct in (100_000, 4_000_000):
    path = os.path.join(tmp, f"junk{distinct}.fastq")
    bases = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (distinct, L), dtype=np.uint8)]
    with open(path, "wb") as f:
        for a in range(0, distinct, 1 << 20):
            rows = bases[a:a + (1 << 20)]
            f.write(b"".join(b"@r\n" + r.tobytes() + b"\n+\n" + b"F" * L + b"\n" for r in rows))
    best = min(cli(path, True, f"junk{distinct}")[0]["unmatched_s"] for _ in range(3))
    print(f"host merge and write, {distinct} distinct windows: unmatched_s best of 3 {best:.4f} s", flush=True)
