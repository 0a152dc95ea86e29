#!/usr/bin/env python3
"""usage: python tools/member_inflate_time.py [n_reads] [rounds] — the CLI on single-member gzip FASTQ
files, with the device ingest (sgc_fastq_stream_submit_member) and with --host-inflate, alternated,
the two tables compared.  Two files of n_reads (default 16.7 M) reads of the bench workload:
  synth     the generator's single-member writer (synth.Sample.write_fastq, reads_per_member = n);
  random_q  the same reads with uniformly random quality characters, compressed with zlib at level 6
            the way pigz does it (one member; 128 KiB parts, each primed with the 32 KiB before it and
            ended with a sync flush, compressed side by side).
Prints the card and its power limit, then one line per run and the best of each."""
import json
import os
import shutil
import struct
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

from sgcount_b200 import synth

N = int(sys.argv[1]) if len(sys.argv) > 1 else 16 << 20
ROUNDS = int(sys.argv[2]) if len(sys.argv) > 2 else 3
BIN = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
SEED = 0xB2000002


def pigz_like(text: bytes, level=6, part=128 << 10) -> bytes:
    parts = [text[i:i + part] for i in range(0, len(text), part)]

    def one(i):
        c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, zlib.Z_DEFAULT_STRATEGY,
                             **({"zdict": text[max(0, i * part - 32768):i * part]} if i else {}))
        return c.compress(parts[i]) + c.flush(zlib.Z_SYNC_FLUSH if i + 1 < len(parts) else zlib.Z_FINISH)

    with ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        body = b"".join(ex.map(one, range(len(parts))))
    crc = 0
    for p in parts:
        crc = zlib.crc32(p, crc)
    return bytes([0x1f, 0x8b, 8, 0, 0, 0, 0, 0, 0, 3]) + body + struct.pack("<II", crc, len(text) & 0xFFFFFFFF)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return "unknown"


def main():
    tmp = tempfile.mkdtemp(prefix="sgc_member_")
    try:
        arr = synth.make_library(SEED, 77441, 20)
        lib = os.path.join(tmp, "lib.fa")
        with open(lib, "wb") as f:
            f.write(b"".join(b">lib.%d\n%s\n" % (i, arr[i].tobytes()) for i in range(len(arr))))
        sample = synth.Sample(SEED, 0, arr, 75, 5, False)
        files = {}
        t0 = time.time()
        files["synth"] = os.path.join(tmp, "synth.fastq.gz")
        sample.write_fastq(files["synth"], 0, N, reads_per_member=N)
        print(f"synth: {N} reads, {os.path.getsize(files['synth']) / 1e6:.0f} MB, one member ({time.time() - t0:.1f} s)", flush=True)
        t0 = time.time()
        text = bytearray(zlib.decompress(open(files["synth"], "rb").read(), 31))
        arr_t = np.frombuffer(text, dtype=np.uint8)
        nl = np.flatnonzero(arr_t == 10)
        # quality lines: line 4r + 3, between newline 4r + 2 and 4r + 3
        starts, ends = nl[2::4] + 1, nl[3::4]
        assert len(starts) == N and np.all(ends - starts == 75)
        rng = np.random.default_rng(7)
        out = arr_t.copy()
        ar = np.arange(75)
        for a in range(0, N, 1 << 20):
            at = (starts[a:a + (1 << 20), None] + ar).ravel()
            out[at] = rng.integers(33, 74, size=len(at), dtype=np.uint8)
        files["random_q"] = os.path.join(tmp, "random_q.fastq.gz")
        with open(files["random_q"], "wb") as f:
            f.write(pigz_like(out.tobytes()))
        del text, arr_t, out
        print(f"random_q: {os.path.getsize(files['random_q']) / 1e6:.0f} MB, one member ({time.time() - t0:.1f} s)", flush=True)
        print(f"card: {card()}", flush=True)
        best = {}
        for name, path in files.items():
            tables = {}
            for r in range(ROUNDS):
                for mode in ("device", "host"):
                    args = [BIN, "-l", lib, "-i", path, "-a", "5", "--timing"] + (["--host-inflate"] if mode == "host" else [])
                    t0 = time.time()
                    p = subprocess.run(args, capture_output=True, text=True)
                    wall = time.time() - t0
                    if p.returncode != 0:
                        raise SystemExit(f"{name} {mode}: exit {p.returncode}\n{p.stderr}")
                    t = json.loads([l for l in p.stderr.splitlines() if l.startswith("{")][-1])
                    tables.setdefault(mode, p.stdout)
                    if p.stdout != tables[mode]:
                        raise SystemExit(f"{name} {mode}: the table changed between runs")
                    print(json.dumps({"file": name, "mode": mode, "round": r, "wall_s": round(wall, 3), "count_s": t["count_s"],
                                      "mreads_per_s": round(N / t["count_s"] / 1e6, 1),
                                      "device_ingest_samples": t["device_ingest_samples"],
                                      "member_pieces": t.get("member_pieces"), "member_chain": t.get("member_chain"),
                                      "member_absorbed": t.get("member_absorbed"), "host_ingest_because": t["host_ingest_because"]}),
                          flush=True)
                    best[(name, mode)] = min(best.get((name, mode), 1e9), t["count_s"])
            same = tables["device"] == tables["host"]
            print(f"{name}: tables identical: {same}", flush=True)
            if not same:
                raise SystemExit(1)
        for (name, mode), s in best.items():
            print(f"best {name} {mode}: count_s {s:.3f}  {N / s / 1e6:.1f} M reads/s")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
