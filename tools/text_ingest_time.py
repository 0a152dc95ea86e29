#!/usr/bin/env python3
"""usage: python tools/text_ingest_time.py [n_reads] [rounds] [--direct-copy-bin PATH] — the CLI on UNCOMPRESSED FASTQ, the device path
(sgc_fastq_stream_submit_text) against --host-inflate (the host reader frames the text), alternated, the
tables and Finished: lines compared across every run.  Samples (seeded, written under a temporary directory
and paged in before anything is timed):
  synth      n_reads (default 16.7 M) reads of the bench workload, the generator's text (constant qualities);
  realistic  the same reads with Phred+33 qualities drawn per position over '#'..'J', 5 % of the quality
             lines starting with '@' and 3 % with '+' (helpers.realistic_fastq's qualities);
  small      the first 4, 16, 64 and 256 MB of synth, cut at a record end: where the host path may win;
  eight      synth under eight names (hard links), default flags against SGC_DEVICE_SAMPLES_IN_FLIGHT=1.
On synth and realistic also the wave sizes 256 MiB and 1 GiB (SGC_TEXT_WAVE; 64 MiB is the default), and with
--direct-copy-bin the CLI of a build with profiles/r9_direct_copy.patch applied (one cudaMemcpyAsync per wave
straight from the mapping, no pinned staging: the rejected pipeline).  Every
run prints one JSON line; per run the best and median count_s and, for the device, text bytes / waves-phase
time as a share of the pinned host-to-device rate measured in the same call (torch, 1 GiB pinned -> device,
best of six).  Exits non-zero when a table or Finished: line differs between runs.  Prints the card, its power limit and clocks before and after; with two devices or more,
also synth on --gpus 2 (else: not measured)."""
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from sgcount_b200 import synth

ARGS = [a for a in sys.argv[1:] if not a.startswith("--")]
DIRECT_BIN = sys.argv[sys.argv.index("--direct-copy-bin") + 1] if "--direct-copy-bin" in sys.argv else None
if DIRECT_BIN:
    ARGS.remove(DIRECT_BIN)
N = int(ARGS[0]) if len(ARGS) > 0 else 16 << 20
ROUNDS = int(ARGS[1]) if len(ARGS) > 1 else 5
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0xB2000019


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return "unknown"


def pinned_rate():
    import torch
    x = torch.empty(1 << 30, dtype=torch.uint8, pin_memory=True)
    y = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    best = 1e9
    for _ in range(6):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        y.copy_(x, non_blocking=True)
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b) / 1e3)
    del x, y
    torch.cuda.empty_cache()
    return (1 << 30) / best


def page_in(paths):
    for p in paths:
        with open(p, "rb") as f:
            while f.read(64 << 20):
                pass


def run(lib, paths, env, extra):
    e = {k: v for k, v in os.environ.items() if not k.startswith("SGC_")}
    e.update(env)
    binary = e.pop("BIN", BIN)
    t0 = time.time()
    p = subprocess.run([binary, "-l", lib, "-i", *paths, "-a", "5", "--timing", *extra], capture_output=True, text=True, env=e)
    wall = time.time() - t0
    if p.returncode != 0:
        raise SystemExit(f"{extra} {env}: exit {p.returncode}\n{p.stderr}")
    fin = [l for l in p.stderr.splitlines() if l.startswith("Finished:")]
    return p.stdout, fin, json.loads([l for l in p.stderr.splitlines() if l.startswith("{")][-1]), wall


def measure(name, lib, paths, runs, rate):
    page_in(paths)
    tables, times, waves = set(), {k: [] for k in runs}, {k: [] for k in runs}
    text = sum(os.path.getsize(p) for p in paths)
    for r in range(ROUNDS):
        for label, (env, extra) in runs.items():
            out, fin, t, wall = run(lib, paths, env, extra)
            tables.add((out, tuple(fin)))
            times[label].append(t["count_s"])
            waves[label].append(t["device_phases_s"][2])
            print(json.dumps({"file": name, "run": label, "round": r, "count_s": t["count_s"], "wall_s": round(wall, 3),
                              "device_phases_s": t["device_phases_s"], "device_ingest_samples": t["device_ingest_samples"],
                              "device_text_bytes": t["device_text_bytes"], "sample_workers": t["sample_workers"],
                              "device_samples_in_flight": t["device_samples_in_flight"], "reads": t["reads"]}), flush=True)
    for label, v in times.items():
        v = sorted(v)
        line = (f"{name} {label}: best {v[0]:.3f} s, median {v[len(v) // 2]:.3f} s over {len(v)} runs, "
                f"{text / v[0] / 1e9:.2f} GB/s of text at best")
        w = sorted(waves[label])
        if w[0] > 0 and len(paths) == 1:
            line += f"; waves phase best {w[0]:.3f} s = {text / w[0] / 1e9:.2f} GB/s, {text / w[0] / rate:.0%} of the pinned copy rate"
        print(line, flush=True)
    print(f"{name}: tables and Finished lines identical across every run: {len(tables) == 1}", flush=True)
    if len(tables) != 1:
        raise SystemExit(f"{name}: the runs disagree on the table or the Finished: lines")


def realistic_text(path, out_path):
    """the synth text with per-position qualities '#'..'J', some lines starting with '@' or '+'"""
    text = np.fromfile(path, dtype=np.uint8)
    nl = np.flatnonzero(text == 10)
    starts, ends = nl[2::4] + 1, nl[3::4]
    assert np.all(ends - starts == 75)
    rng = np.random.default_rng(SEED + 1)
    ar = np.arange(75)
    for a in range(0, len(starts), 1 << 20):
        s = starts[a:a + (1 << 20)]
        at = (s[:, None] + ar).ravel()
        text[at] = rng.integers(ord("#"), ord("J") + 1, size=len(at), dtype=np.uint8)
        first = rng.random(len(s))
        text[s[first < 0.05]] = ord("@")
        text[s[(first >= 0.05) & (first < 0.08)]] = ord("+")
    text.tofile(out_path)
    return nl


def main():
    tmp = tempfile.mkdtemp(prefix="sgc_text_ingest_")
    try:
        rate = pinned_rate()
        print(f"card: {card()}; host cores: {os.cpu_count()}; {N} reads; {ROUNDS} runs each; "
              f"pinned host-to-device copy (1 GiB, torch, best of 6): {rate / 1e9:.1f} GB/s", flush=True)
        arr = synth.make_library(SEED, 77441, 20)
        lib = os.path.join(tmp, "lib.fa")
        with open(lib, "wb") as f:
            f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
        synth_path = os.path.join(tmp, "synth.fastq")
        synth.Sample(SEED, 0, arr, 75, 5, False).write_fastq(synth_path, 0, N, gz_level=0)
        real_path = os.path.join(tmp, "realistic.fastq")
        nl = realistic_text(synth_path, real_path)
        host = ({}, ["--host-inflate"])
        ab = {"device": ({}, []), "host": host,
              **({"direct_copy": ({"BIN": DIRECT_BIN}, [])} if DIRECT_BIN else {}),
              "wave_256M": ({"SGC_TEXT_WAVE": str(256 << 20)}, []), "wave_1G": ({"SGC_TEXT_WAVE": str(1 << 30)}, [])}
        for name, path in (("synth", synth_path), ("realistic", real_path)):
            print(f"{name}: {os.path.getsize(path) / 1e6:.0f} MB", flush=True)
            measure(name, lib, [path], ab, rate)
        os.remove(real_path)
        ends = nl[3::4] + 1
        for mb in (4, 16, 64, 256):
            cut = int(ends[np.searchsorted(ends, mb * 1000000)])
            small = os.path.join(tmp, f"small_{mb}.fastq")
            with open(synth_path, "rb") as f, open(small, "wb") as g:
                g.write(f.read(cut))
            measure(f"small_{mb}MB", lib, [small], {"device": ({}, []), "host": host}, rate)
            os.remove(small)
        paths = []
        for i in range(8):
            paths.append(os.path.join(tmp, f"eight_{i}.fastq"))
            os.link(synth_path, paths[-1])
        measure("eight", lib, paths, {"default": ({}, []), "one": ({"SGC_DEVICE_SAMPLES_IN_FLIGHT": "1"}, [])}, rate)
        gpus = int(subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.count("GPU "))
        if gpus >= 2:
            measure("synth_gpus2", lib, [synth_path], {"one": ({}, []), "two": ({}, ["--gpus", "2"])}, rate)
        else:
            print("several devices: not measured (one device in this box)", flush=True)
        print(f"card: {card()}", flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
