#!/usr/bin/env python3
"""usage: python tools/member_samples_time.py [n_reads] [rounds] — the CLI on EIGHT single-member gzip FASTQ
samples at once, with the samples side by side on the one device and one at a time, alternated, the tables
compared.  Two kinds of sample, each of n_reads (default 16.7 M) reads of the bench workload, built by
tools/multi_member_time.py's generators:
  synth     the generator's single-member writer (249 MB at 16.7 M reads);
  random_q  the same reads with uniformly random quality characters, compressed at level 6 the way pigz
            does it (1155 MB).
The eight samples of a kind are hard links to one file under eight names (the reads are the same; the
CLI reads, maps and decodes each as its own sample).  Runs, alternated within each round:
  default   the CLI's own choice (four per device when every sample is device-bound);
  one       SGC_DEVICE_SAMPLES_IN_FLIGHT=1: one sample at a time on the device;
  two       SGC_DEVICE_SAMPLES_IN_FLIGHT=2;
  eight     SGC_DEVICE_SAMPLES_IN_FLIGHT=8;
  host_t8   --host-inflate -t 8: eight samples inflated on the host side by side.
Prints the card, its power limit and clocks (before and after), one line per run, and per run best and
median count_s and whether every table of a kind is identical."""
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from member_inflate_time import card, pigz_like
from multi_member_time import N, SEED, random_q_text
from sgcount_b200 import synth

ROUNDS = int(sys.argv[2]) if len(sys.argv) > 2 else 3
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SAMPLES = 8
RUNS = {"default": ({}, []), "one": ({"SGC_DEVICE_SAMPLES_IN_FLIGHT": "1"}, []), "two": ({"SGC_DEVICE_SAMPLES_IN_FLIGHT": "2"}, []),
        "eight": ({"SGC_DEVICE_SAMPLES_IN_FLIGHT": "8"}, []), "host_t8": ({}, ["--host-inflate", "-t", "8"])}


def run(lib, paths, env, extra):
    e = {k: v for k, v in os.environ.items() if not k.startswith("SGC_")}
    e.update(env)
    t0 = time.time()
    p = subprocess.run([BIN, "-l", lib, "-i", *paths, "-a", "5", "--timing", *extra], capture_output=True, text=True, env=e)
    wall = time.time() - t0
    if p.returncode != 0:
        raise SystemExit(f"{extra} {env}: exit {p.returncode}\n{p.stderr}")
    fin = [l for l in p.stderr.splitlines() if l.startswith("Finished:")]
    return p.stdout, fin, json.loads([l for l in p.stderr.splitlines() if l.startswith("{")][-1]), wall


def measure(name, lib, paths):
    tables, times = set(), {k: [] for k in RUNS}
    for r in range(ROUNDS):
        for label, (env, extra) in RUNS.items():
            out, fin, t, wall = run(lib, paths, env, extra)
            tables.add((out, tuple(fin)))
            times[label].append(t["count_s"])
            print(json.dumps({"file": name, "run": label, "round": r, "count_s": t["count_s"], "wall_s": round(wall, 3),
                              "sample_workers": t["sample_workers"], "ingest_threads": t["ingest_threads"],
                              "device_ingest_samples": t["device_ingest_samples"],
                              "device_samples_in_flight": t["device_samples_in_flight"], "reads": t["reads"]}), flush=True)
    for label, v in times.items():
        v = sorted(v)
        print(f"{name} {label}: best {v[0]:.3f} s, median {v[len(v) // 2]:.3f} s over {len(v)} rounds, "
              f"{SAMPLES * N / v[0] / 1e6:.1f} M reads/s at best", flush=True)
    print(f"{name}: tables and Finished lines identical across every run: {len(tables) == 1}", flush=True)


def main():
    tmp = tempfile.mkdtemp(prefix="sgc_member_samples_")
    try:
        print(f"card: {card()}; host cores: {os.cpu_count()}; {SAMPLES} samples of {N} reads; {ROUNDS} rounds", flush=True)
        arr = synth.make_library(SEED, 77441, 20)
        lib = os.path.join(tmp, "lib.fa")
        with open(lib, "wb") as f:
            f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
        sample = synth.Sample(SEED, 0, arr, 75, 5, False)
        for name in ("synth", "random_q"):
            base = os.path.join(tmp, f"{name}.fastq.gz")
            if name == "synth":
                sample.write_fastq(base, 0, N, reads_per_member=N)
            else:
                out, _ = random_q_text(sample, os.path.join(tmp, "x.fastq.gz"))
                with open(base, "wb") as f:
                    f.write(pigz_like(out.tobytes()))
                del out
                os.remove(os.path.join(tmp, "x.fastq.gz"))
            paths = []
            for i in range(SAMPLES):
                paths.append(os.path.join(tmp, f"{name}_{i}.fastq.gz"))
                os.link(base, paths[-1])
            print(f"{name}: {os.path.getsize(base) / 1e6:.0f} MB a sample, one member", flush=True)
            measure(name, lib, paths)
            for p in paths + [base]:
                os.remove(p)
        print(f"card: {card()}", flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
