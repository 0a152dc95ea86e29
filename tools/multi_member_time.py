#!/usr/bin/env python3
"""usage: python tools/multi_member_time.py [n_reads] [rounds] [parent_sgcount|-] [sections] [members] — the CLI on gzip FASTQ files
of M in {1, 2, 4, 8, 32} members (not BGZF), with the device ingest (sgc_fastq_stream_submit_gzip; M = 1:
sgc_fastq_stream_submit_member) and with --host-inflate at the default ingest threads and at
--ingest-threads 2 and 4, alternated, the tables compared.  SGC_MULTI_MEMBER_DEVICE=1 sends every file to
the device whatever the routing would do; one run without it records what the CLI picks.  The files hold
the same n_reads (default 16.7 M) reads of the bench workload:
  synth     the generator's writer (synth.Sample.write_fastq, reads_per_member = n / M);
  random_q  the same reads with uniformly random quality characters, cut into M members at record
            boundaries, each compressed with zlib at level 6 the way pigz does it
            (tools/member_inflate_time.py).
Then the size floor: synth files of two members and fewer reads, device against the host.  With
parent_sgcount (the CLI built from the parent commit), single-member device timings of both builds,
alternated.  `sections` (default synth,random_q,floor,regress) picks the parts to run, `members` (comma-separated)
the member counts.  Prints the card, its power
limit and clocks, one line per run and the best of each."""
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np

from member_inflate_time import card, pigz_like
from sgcount_b200 import synth

N = int(sys.argv[1]) if len(sys.argv) > 1 else 16 << 20
ROUNDS = int(sys.argv[2]) if len(sys.argv) > 2 else 2
PARENT = sys.argv[3] if len(sys.argv) > 3 and sys.argv[3] != "-" else None
SECTIONS = sys.argv[4].split(",") if len(sys.argv) > 4 else ["synth", "random_q", "floor", "regress"]
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0xB2000002
MEMBERS = [int(m) for m in sys.argv[5].split(",")] if len(sys.argv) > 5 else [1, 2, 4, 8, 32]
MODES = {"device": [], "host": ["--host-inflate"], "host_t2": ["--host-inflate", "--ingest-threads", "2"],
         "host_t4": ["--host-inflate", "--ingest-threads", "4"]}


def run(bin_path, lib, path, extra, force):
    env = dict(os.environ)
    env.pop("SGC_MULTI_MEMBER_DEVICE", None)
    if force:
        env["SGC_MULTI_MEMBER_DEVICE"] = "1"
    t0 = time.time()
    p = subprocess.run([bin_path, "-l", lib, "-i", path, "-a", "5", "--timing"] + extra, capture_output=True, text=True, env=env)
    wall = time.time() - t0
    if p.returncode != 0:
        raise SystemExit(f"{path} {extra}: exit {p.returncode}\n{p.stderr}")
    return p.stdout, json.loads([l for l in p.stderr.splitlines() if l.startswith("{")][-1]), wall


def line(**kw):
    print(json.dumps(kw), flush=True)


def measure(name, m, n, lib, path, best, modes=MODES, rounds=ROUNDS):
    tables = {}
    for r in range(rounds):
        for mode, extra in modes.items():
            out, t, wall = run(BIN, lib, path, extra, mode == "device")
            tables.setdefault(mode, out)
            if out != tables[mode]:
                raise SystemExit(f"{name} M={m} {mode}: the table changed between runs")
            line(file=name, members=m, reads=n, mode=mode, round=r, wall_s=round(wall, 3), count_s=t["count_s"],
                 mreads_per_s=round(n / t["count_s"] / 1e6, 1), device_ingest_samples=t["device_ingest_samples"],
                 gzip_members=t["gzip_members"], member_pieces=t["member_pieces"], member_chain=t["member_chain"],
                 ingest_threads=t["ingest_threads"], host_ingest_because=t["host_ingest_because"])
            key = (name, m, n, mode)
            best[key] = min(best.get(key, 1e9), t["count_s"])
    _, t, _ = run(BIN, lib, path, [], False)
    line(file=name, members=m, reads=n, mode="routed", device_ingest_samples=t["device_ingest_samples"],
         ingest_threads=t["ingest_threads"], host_ingest_because=t["host_ingest_because"])
    same = len(set(tables.values())) == 1
    print(f"{name} M={m} reads={n}: tables identical across device and host runs: {same}", flush=True)
    if not same:
        raise SystemExit(1)


def random_q_text(sample, path):
    """the text of the single-member synthetic file with uniformly random quality characters, and where
    every record ends"""
    sample.write_fastq(path, 0, N, reads_per_member=N)
    text = np.frombuffer(zlib.decompress(open(path, "rb").read(), 31), dtype=np.uint8)
    nl = np.flatnonzero(text == 10)
    starts, ends = nl[2::4] + 1, nl[3::4]
    assert len(starts) == N and np.all(ends - starts == 75)
    rng = np.random.default_rng(7)
    out = text.copy()
    ar = np.arange(75)
    for a in range(0, N, 1 << 20):
        at = (starts[a:a + (1 << 20), None] + ar).ravel()
        out[at] = rng.integers(33, 74, size=len(at), dtype=np.uint8)
    return out, np.concatenate([[0], nl[3::4] + 1])


def main():
    tmp = tempfile.mkdtemp(prefix="sgc_multi_member_")
    try:
        print(f"card: {card()}", flush=True)
        print(f"host cores: {os.cpu_count()}", flush=True)
        arr = synth.make_library(SEED, 77441, 20)
        lib = os.path.join(tmp, "lib.fa")
        with open(lib, "wb") as f:
            f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
        sample = synth.Sample(SEED, 0, arr, 75, 5, False)
        best = {}
        path = os.path.join(tmp, "x.fastq.gz")
        for m in MEMBERS if "synth" in SECTIONS else ():
            sample.write_fastq(path, 0, N, reads_per_member=(N + m - 1) // m)
            print(f"synth M={m}: {os.path.getsize(path) / 1e6:.0f} MB", flush=True)
            measure("synth", m, N, lib, path, best)
        if "random_q" in SECTIONS:
            out, record_end = random_q_text(sample, path)
            for m in MEMBERS:
                cuts = [int(record_end[(N * i) // m]) for i in range(m + 1)]
                with open(path, "wb") as f:
                    for i in range(m):
                        f.write(pigz_like(out[cuts[i]:cuts[i + 1]].tobytes()))
                print(f"random_q M={m}: {os.path.getsize(path) / 1e6:.0f} MB", flush=True)
                measure("random_q", m, N, lib, path, best)
            del out
        # the size floor: two members, fewer reads
        for n in (1 << 18, 1 << 20, 1 << 21, 1 << 22) if "floor" in SECTIONS else ():
            sample.write_fastq(path, 0, n, reads_per_member=(n + 1) // 2)
            print(f"floor synth M=2 reads={n}: {os.path.getsize(path) / 1e6:.1f} MB", flush=True)
            measure("synth", 2, n, lib, path, best, {k: MODES[k] for k in ("device", "host", "host_t2")}, max(ROUNDS, 3))
        for (name, m, n, mode), s in sorted(best.items()):
            print(f"best {name} M={m} reads={n} {mode}: count_s {s:.3f}  {n / s / 1e6:.1f} M reads/s")
        # one member: this build against the parent's, alternated
        if PARENT and "regress" in SECTIONS:
            files = {"synth": os.path.join(tmp, "synth1.fastq.gz"), "random_q": os.path.join(tmp, "random_q1.fastq.gz")}
            sample.write_fastq(files["synth"], 0, N, reads_per_member=N)
            out, _ = random_q_text(sample, path)
            with open(files["random_q"], "wb") as f:
                f.write(pigz_like(out.tobytes()))
            del out
            for name, p in files.items():
                res = {}
                for r in range(ROUNDS):
                    for build, b in (("this", BIN), ("parent", PARENT)):
                        o, t, _ = run(b, lib, p, [], False)
                        res.setdefault(build, []).append((t["count_s"], o))
                        line(file=name, members=1, build=build, round=r, count_s=t["count_s"],
                             device_ingest_samples=t["device_ingest_samples"])
                same = len({o for v in res.values() for _, o in v}) == 1
                cs = {k: sorted(c for c, _ in v) for k, v in res.items()}
                print(f"single member {name}: this best {cs['this'][0]:.3f} s median {cs['this'][len(cs['this']) // 2]:.3f} s, "
                      f"parent best {cs['parent'][0]:.3f} s median {cs['parent'][len(cs['parent']) // 2]:.3f} s; "
                      f"tables identical: {same}", flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
