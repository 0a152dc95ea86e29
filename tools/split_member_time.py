#!/usr/bin/env python3
"""usage: python tools/split_member_time.py [n_reads] [rounds] [big_reads] [parent_bin] [files] — the CLI on one plain
gzip FASTQ decoded by one stream (today's path) against several streams together (SGC_MEMBER_LANES,
sgc_fastq_stream_submit_gzip_split), alternated, every table compared with the first.  Files: the two of
tools/member_inflate_time.py at n_reads (default 16.7 M: `synth`, and `random_q`, random qualities at
level 6 written the way pigz does), and `big`, big_reads (default 134 M) synthetic reads in members of
n_reads (the generator writes at most 4 GiB of text per member), whose text spans several waves of one
stream; it goes to the device whatever its member count (SGC_MULTI_MEMBER_DEVICE).  `files`: a comma
list of the three names (default all).  Configurations:
  parent    parent_bin (a build of the parent commit), one stream, when given;
  lanes1    this build, one stream;
  lanes2    two streams on one device;
  gpusN     N streams on N devices (--gpus N), for every N from 2 up to min(8, devices).
Prints the card and its power limit, one line per run, and the best and the median of each."""
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np

from member_inflate_time import SEED, card, pigz_like
from sgcount_b200 import synth

N = int(sys.argv[1]) if len(sys.argv) > 1 else 16 << 20
ROUNDS = int(sys.argv[2]) if len(sys.argv) > 2 else 5
BIG = int(sys.argv[3]) if len(sys.argv) > 3 else 134 << 20
PARENT = sys.argv[4] if len(sys.argv) > 4 else ""
FILES = sys.argv[5].split(",") if len(sys.argv) > 5 else ["synth", "random_q", "big"]
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")


def devices():
    p = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True)
    return max(1, len([l for l in p.stdout.splitlines() if l.startswith("GPU ")]))


def random_q(path_in, path_out):
    text = np.frombuffer(zlib.decompress(open(path_in, "rb").read(), 31), dtype=np.uint8)
    nl = np.flatnonzero(text == 10)
    starts = nl[2::4] + 1
    out = text.copy()
    rng = np.random.default_rng(7)
    ar = np.arange(75)
    for a in range(0, len(starts), 1 << 20):
        at = (starts[a:a + (1 << 20), None] + ar).ravel()
        out[at] = rng.integers(33, 74, size=len(at), dtype=np.uint8)
    with open(path_out, "wb") as f:
        f.write(pigz_like(out.tobytes()))


def main():
    tmp = tempfile.mkdtemp(prefix="sgc_split_")
    try:
        arr = synth.make_library(SEED, 77441, 20)
        lib = os.path.join(tmp, "lib.fa")
        with open(lib, "wb") as f:
            f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
        sample = synth.Sample(SEED, 0, arr, 75, 5, False)
        files, reads = {}, {}
        for name, n in (("synth", N), ("big", BIG)):
            if name not in FILES and not (name == "synth" and "random_q" in FILES):
                continue
            t0 = time.time()
            files[name], reads[name] = os.path.join(tmp, f"{name}.fastq.gz"), n
            sample.write_fastq(files[name], 0, n, reads_per_member=N)
            print(f"{name}: {n} reads, {os.path.getsize(files[name]) / 1e6:.0f} MB, {(n + N - 1) // N} member(s) ({time.time() - t0:.1f} s)",
                  flush=True)
        if "random_q" in FILES:
            t0 = time.time()
            files["random_q"], reads["random_q"] = os.path.join(tmp, "random_q.fastq.gz"), N
            random_q(files["synth"], files["random_q"])
            print(f"random_q: {os.path.getsize(files['random_q']) / 1e6:.0f} MB, one member ({time.time() - t0:.1f} s)", flush=True)
        n_dev = devices()
        print(f"card: {card()}; devices: {n_dev}", flush=True)
        configs = ([("parent", PARENT, {}, [])] if PARENT else []) + [("lanes1", BIN, {}, []), ("lanes2", BIN, {"SGC_MEMBER_LANES": "2"}, [])]
        configs += [(f"gpus{g}", BIN, {"SGC_MEMBER_LANES": str(g)}, ["--gpus", str(g)]) for g in range(2, min(8, n_dev) + 1)]
        times = {}
        for name in FILES:
            table = None
            for r in range(ROUNDS):
                for label, exe, env, extra in configs:
                    args = [exe, "-l", lib, "-i", files[name], "-a", "5", "--timing"] + extra
                    big = {"SGC_MULTI_MEMBER_DEVICE": "1"} if name == "big" else {}
                    p = subprocess.run(args, capture_output=True, text=True, env={**os.environ, **env, **big})
                    if p.returncode != 0:
                        raise SystemExit(f"{name} {label}: exit {p.returncode}\n{p.stderr}")
                    t = json.loads([l for l in p.stderr.splitlines() if l.startswith("{")][-1])
                    table = table or p.stdout
                    if p.stdout != table:
                        raise SystemExit(f"{name} {label}: the table differs")
                    print(json.dumps({"file": name, "config": label, "round": r, "count_s": t["count_s"],
                                      "device_ingest_samples": t["device_ingest_samples"], "member_lanes": t.get("member_lanes"),
                                      "read_shards_per_sample": t["read_shards_per_sample"], "member_chain": t["member_chain"],
                                      "device_phases_s": t["device_phases_s"]}), flush=True)
                    times.setdefault((name, label), []).append(t["count_s"])
            print(f"{name}: tables identical: True", flush=True)
        for (name, label), v in times.items():
            print(f"{name:9s} {label:7s} best {min(v):.3f} s  median {statistics.median(v):.3f} s  "
                  f"{reads[name] / min(v) / 1e6:.1f} M reads/s")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
