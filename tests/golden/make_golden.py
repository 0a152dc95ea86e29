#!/usr/bin/env python3
"""Derives the config-1 golden fixtures from the reference's example data.

Run with the example/ directory of the reference's source tree (the tests read only the
committed outputs):   python tests/golden/make_golden.py <sgcount source>/example

Outputs, all under tests/golden/:
  example/<name>.gz          the example FASTA/FASTQ records re-serialised (id, seq, +, qual)
                             and re-compressed with mtime=0 -- record content is unchanged
  example/g2s.txt            gene map, verbatim
  example/expected.json      matcher-INDEPENDENT known answers: every example read header
                             is `@seq.<guide sequence>.<n>` (or `@nonsense`), so the header
                             names the guide the read was simulated from.  The expected
                             table is a tally of those labels, not the output of any matcher.

The reference has no test that pins these files (SURVEY.md §4); the labels are the strongest
pin available without a Rust toolchain.
"""
import gzip
import hashlib
import json
import os
import shutil
import sys

DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "example")

FASTQ = ["sequence", "zero.sequence", "diff.sequence", "offset", "offset_clipped"]
K = 20
OFFSET = 5


def read_records(path):
    with gzip.open(path, "rb") as f:
        lines = f.read().split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    step = 4 if lines[0].startswith(b"@") else 2
    return [lines[i:i + step] for i in range(0, len(lines), step)]


def write_gz(path, records):
    raw = b"".join(b"\n".join(r) + b"\n" for r in records)
    with open(path, "wb") as f, gzip.GzipFile(fileobj=f, mode="wb", mtime=0, filename="") as g:
        g.write(raw)


def main():
    if len(sys.argv) != 2:
        raise SystemExit("usage: make_golden.py <reference example directory>")
    src = sys.argv[1]
    os.makedirs(DST, exist_ok=True)
    lib = read_records(os.path.join(src, "library.fasta.gz"))
    write_gz(os.path.join(DST, "library.fasta.gz"), lib)
    shutil.copyfile(os.path.join(src, "g2s.txt"), os.path.join(DST, "g2s.txt"))
    seq_to_alias = {r[1].decode(): r[0][1:].decode() for r in lib}
    aliases = [r[0][1:].decode() for r in lib]

    expected = {"library": {"n": len(lib), "k": K, "aliases": aliases}, "offset": OFFSET, "fixtures": {}}
    for name in FASTQ:
        recs = read_records(os.path.join(src, name + ".fastq.gz"))
        write_gz(os.path.join(DST, name + ".fastq.gz"), recs)
        counts = {a: 0 for a in aliases}
        labelled = clipped = 0
        for r in recs:
            hdr, seq = r[0].decode(), r[1]
            if hdr.startswith("@seq."):
                guide = hdr.split(".")[1]
                # a read too short to hold offset+K bases cannot be trimmed (counter.rs:175)
                if len(seq) < OFFSET + K:
                    clipped += 1
                    continue
                counts[seq_to_alias[guide]] += 1
                labelled += 1
        rows = "\n".join(f"{a}\t{c}" for a, c in sorted(counts.items()))
        expected["fixtures"][name] = {
            "total_reads": len(recs),
            "matched_reads": labelled,
            "clipped_reads": clipped,
            "first_len": len(recs[0][1]),
            "min_len": min(len(r[1]) for r in recs),
            "max_len": max(len(r[1]) for r in recs),
            "counts": [counts[a] for a in aliases],
            "sha256_16": hashlib.sha256(rows.encode()).hexdigest()[:16],
        }
    with open(os.path.join(DST, "expected.json"), "w") as f:
        json.dump(expected, f, indent=1)
    for name, fx in expected["fixtures"].items():
        print(name, fx["total_reads"], fx["matched_reads"], fx["sha256_16"])


if __name__ == "__main__":
    main()
