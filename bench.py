#!/usr/bin/env python3
"""bench.py — reads/sec of the sgcount match-and-count path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], the configuration the metric is quoted on): Brunello-
shaped synthetic library (77 441 x 20 bp, seed 0xB2000002), one sample of 50 M x 75 bp reads,
one-mismatch table on, Forward(5).  A step is one pass of the hot path over the whole sample.
With N > 1 (torchrun) every rank holds its own 50 M-read shard of an N x 50 M-read sample (weak
scaling) and the per-guide count vectors are summed with an NCCL all-reduce inside the step.

Printed JSON (rank 0, one line):
  value      kernel-only reads/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        the same through sgc_counter_submit with PINNED HOST buffers: H2D copies of the
             sequence lines and the D2H read-back of the count vector are inside the timed region;
             e2e.roofline puts it against the host->device copy rate measured in the same run
  roofline   algorithmic bytes (read_len+1 per read) / mean duration of the count launches
             against the measured HBM copy peak of MEASURED_PEAKS.json
  configs    the other BASELINE configs at their FULL sizes, generated in HBM, kernel-timed:
             c1 the example fixture; c3 GeCKO-shaped, 4 samples x 100 M, offsets detected;
             c4 CRISPRi-shaped, 8 samples x 200 M, sample-sharded over the ranks (strong scaling);
             c5 one 1 B-read sample in 8 read shards over the ranks + the count reduce
  parity / parity_n   the GPU tables of this very run against the oracle on read prefixes
             (rank 0, every N; the oracle is the checker, never the thing measured)
  cpu_baseline  the oracle port of the reference's loop on this box's host cores (N = 1 only)
"""
import argparse
import ctypes
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SEED = 0xB2000002
N_GUIDES = 77441
K = 20
READ_LEN = 75
STRIDE = READ_LEN + 1
OFFSET = 5
READS_PER_GPU = 50_000_000
WORKLOAD = "config2: Brunello-shaped 77441x20bp library, 1 sample x 50M x 75bp reads, 1-mismatch, Forward(5)"
FALLBACK_HBM_GBS = 6650.0
PARITY_PREFIX = 1_000_000  # reads per shard the oracle re-counts

# BASELINE.json configs 3-5 (SURVEY.md §8d).  sample = (sample index, reverse, offset).
CONFIGS = {
    "c3": {"what": "config3: GeCKO-v2-shaped 123411x20bp library, 4 samples x 100M x 75bp reads, offsets detected "
                   "(truth F0 R12 F23 R5), sharded by sample",
           "seed": 0xB2000003, "n_guides": 123411, "reads_per_sample": 100_000_000, "shards_per_sample": 1,
           "samples": [(0, False, 0), (1, True, 12), (2, False, 23), (3, True, 5)]},
    "c4": {"what": "config4: CRISPRi-shaped 200000x20bp library (20000 genes), 8 samples x 200M x 75bp reads, offsets "
                   "detected, sharded by sample, count table summed over the ranks",
           "seed": 0xB2000004, "n_guides": 200000, "reads_per_sample": 200_000_000, "shards_per_sample": 1,
           "samples": [(0, False, 7), (1, True, 30), (2, False, 0), (3, True, 12), (4, False, 23), (5, True, 5),
                       (6, False, 15), (7, True, 40)]},
    "c5": {"what": "config5: config-4 library, ONE sample of 1B x 75bp reads in 8 read shards of 125M, offset detected "
                   "once, count vectors reduced",
           "seed": 0xB2000004, "n_guides": 200000, "reads_per_sample": 1_000_000_000, "shards_per_sample": 8,
           "samples": [(100, False, 9)]},
}


def cpu_threads() -> int:
    try:
        return max(1, min(len(os.sched_getaffinity(0)), 64))
    except AttributeError:
        return max(1, min(os.cpu_count() or 1, 64))


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def bench_config(world: int, reads_per_gpu: int) -> dict:
    """`config` of the JSON line: the same dict in both arms (--impl b200 / reference)."""
    return {
        "workload": WORKLOAD,
        "n_guides": N_GUIDES,
        "guide_len": K,
        "read_len": READ_LEN,
        "reads_per_gpu": reads_per_gpu,
        "l2": "inputs (3.8 GB per step) are larger than L2; no flush needed",
        "parallelism": (f"read-sharded x{world}, NCCL all-reduce of u64[{N_GUIDES + 2}] per step on a second stream, "
                        "overlapping the next step's kernel") if world > 1 else "1 GPU",
    }


def library_fasta(lib_arr) -> bytes:
    return b"".join(b">lib.%d\n%s\n" % (i, lib_arr[i].tobytes()) for i in range(len(lib_arr)))


def dump_outputs(out_dir, counts, total, matched):
    """--dump-outputs: what Counter.finish() handed back after the last timed step, so that two
    builds can be compared output for output on the same seeded sample.  float64 holds every count
    exactly (all are below 2**53); the three arrays hold (N_GUIDES + 2) x 8 bytes."""
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("counts", counts), ("total_reads", [total]), ("matched_reads", [matched])):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(arr, dtype=np.float64))


# ---------------------------------------------------------------------------------------------
# oracle leg: cpu_baseline of the GPU arm, the whole `--impl reference` arm, and the parity checker
# ---------------------------------------------------------------------------------------------
class OracleLeg:
    """The reference is Rust and cannot be built in this image, so the CPU comparator is the
    oracle port (oracle/oracle.cpp): byte-string hash maps, literal Permuter, one token per
    probe.  The reference parallelises over samples only (count.rs:117-136); with one sample
    it is single-threaded.  We give it every host thread by sharding the sample's reads, which
    the reference itself cannot do — the number is generous to the CPU side."""

    def __init__(self, lib_arr, sample_reads: int, threads: int):
        from oracle import oracle as orc
        from sgcount_b200 import synth

        self.orc = orc
        self.threads = threads
        self.n = sample_reads
        recs = orc.Records.from_bytes(library_fasta(lib_arr))
        self.lib_records = recs
        self.library = orc.Library.from_reader(recs)
        t0 = time.perf_counter()
        self.permuter = orc.Permuter.new(self.library)
        self.permuter_s = time.perf_counter() - t0
        sample = synth.Sample(SEED, 0, lib_arr, READ_LEN, OFFSET, False)
        self.lines = sample.fill_host(0, sample_reads)
        off = np.arange(0, self.lines.nbytes + 1, STRIDE, dtype=np.uint64)
        self.records = orc.Records.from_lines(self.lines, off)

    def step(self, threads=None, n=None):
        recs = self.records
        if n is not None and n < self.n:
            recs = self.orc.Records.from_lines(self.lines[:n * STRIDE], np.arange(0, n * STRIDE + 1, STRIDE, dtype=np.uint64))
        t0 = time.perf_counter()
        c = self.orc.Counter.new(recs, self.library, self.permuter, self.orc.Offset.Forward(OFFSET),
                                 None, True, n_threads=threads or self.threads)
        dt = time.perf_counter() - t0
        return dt, c

    def describe(self):
        return (f"first {self.n} reads of the workload's sample 0, pre-parsed in memory, read-sharded over "
                f"{self.threads} threads; one-off Permuter::new took {self.permuter_s:.1f} s on 1 thread (not timed)")


# ---------------------------------------------------------------------------------------------
# end to end from a gzip FASTQ through the C++ host (ingest + count + table), with the oracle's
# gunzip + parse + match on the same file beside it
# ---------------------------------------------------------------------------------------------
def run_cli(exe, lib_path, fq_paths, extra, out_path):
    import subprocess

    best = None
    for _ in range(3):  # the first run pages the file in; a box of this pool varies from run to run (profiles/r2e_cli_ab.txt)
        t0 = time.perf_counter()
        p = subprocess.run([exe, "-l", lib_path, "-i", *fq_paths, "-q", "-o", out_path, "--timing", *extra],
                           capture_output=True, text=True, timeout=900)
        wall = time.perf_counter() - t0
        if p.returncode != 0:
            return None, "sgcount failed: " + p.stderr.strip()[-300:]
        timing = json.loads([l for l in p.stderr.splitlines() if l.startswith("{")][-1])
        if best is None or timing["count_s"] < best[0]["count_s"]:
            best = (timing, wall)
    return best, None


def fastq_leg(lib_arr, n_reads: int, with_oracle: bool, gpus: int = 1):
    """N = 1: the CLI on one multi-member gzip FASTQ, oracle beside it.  N > 1 (run by rank 0 while
    the other ranks wait): the same ONE sample with --gpus 1 and with --gpus N (read shards over
    the devices, sgc_reduce_counts); the two tables must be identical."""
    import shutil
    import tempfile

    from sgcount_b200 import synth

    exe = os.path.join(ROOT, "sgcount_b200", "lib", "sgcount")
    if not os.path.exists(exe):
        return {"unavailable": "sgcount host binary not built"}
    tmp = tempfile.mkdtemp(prefix="sgc_bench_")
    try:
        lib_path = os.path.join(tmp, "library.fa")
        with open(lib_path, "wb") as f:
            f.write(library_fasta(lib_arr))
        fq = os.path.join(tmp, "sample0.fastq.gz")
        sample = synth.Sample(SEED, 0, lib_arr, READ_LEN, OFFSET, False)
        sample.write_fastq(fq, 0, n_reads, reads_per_member=1 << 20, gz_level=1)
        gz_bytes = os.path.getsize(fq)
        out_path = os.path.join(tmp, "counts.tsv")
        best, err = run_cli(exe, lib_path, [fq], ["-a", str(OFFSET)], out_path)
        if err:
            return {"unavailable": err}
        timing, wall = best
        text_one = open(out_path).read()
        rows = text_one.rstrip("\n").split("\n")
        table = {r.split("\t")[0]: int(r.split("\t")[1]) for r in rows[1:]}
        res = {"value": timing["reads"] / timing["count_s"], "unit": "reads/s", "reads": timing["reads"],
               "count_s": timing["count_s"], "process_wall_s": wall, "gz_bytes": gz_bytes,
               "ingest_threads": timing["ingest_threads"],
               "members": (n_reads + (1 << 20) - 1) >> 20,
               "what": "sgcount CLI on a multi-member gzip FASTQ (1 Mi reads per member, so at most `members` inflate "
                       "threads have work): member-parallel inflate + record framing, H2D, count kernel, D2H; table "
                       "build and process start-up are outside count_s"}
        # the same reads as BGZF (bgzip's blocked gzip, 64 KB blocks cut anywhere): the CLI inflates,
        # frames and counts such a file on the device (sgc_fastq_stream_*), no host core in the loop
        bgzf = os.path.join(tmp, "sample0.bgzf.fastq.gz")
        sample.write_fastq_bgzf(bgzf, 0, n_reads, gz_level=1)
        out_d = os.path.join(tmp, "counts_dev.tsv")
        best_d, err_d = run_cli(exe, lib_path, [bgzf], ["-a", str(OFFSET)], out_d)
        if err_d:
            res["device_ingest"] = {"unavailable": err_d}
        else:
            td, wd = best_d
            same = open(out_d).read().replace("sample0.bgzf", "sample0") == text_one
            res["device_ingest"] = {"value": td["reads"] / td["count_s"], "unit": "reads/s", "count_s": td["count_s"],
                                    "process_wall_s": wd, "gz_bytes": os.path.getsize(bgzf), "blocks": td.get("device_blocks"),
                                    "device_ingest_samples": td.get("device_ingest_samples"), "same_table": same,
                                    "what": "the same reads as a BGZF file through the same CLI: one device thread inflates "
                                            "each 64 KB block, a newline scan frames the records, the guide-window spans are "
                                            "cut out and counted; only the compressed bytes cross PCIe"}
            assert same, "device ingest table differs from the host path's"
            best_h, err_h = run_cli(exe, lib_path, [bgzf], ["-a", str(OFFSET), "--host-inflate"], out_d)
            if not err_h:
                res["device_ingest"]["host_inflate_same_file"] = {"value": best_h[0]["reads"] / best_h[0]["count_s"],
                                                                  "unit": "reads/s", "count_s": best_h[0]["count_s"]}
        if gpus > 1:
            out_n = os.path.join(tmp, "counts_n.tsv")
            best, err = run_cli(exe, lib_path, [fq], ["-a", str(OFFSET), "--gpus", str(gpus), "--read-shards", str(gpus)], out_n)
            if err:
                res["read_sharded"] = {"unavailable": err}
            else:
                tn, wn = best
                same = open(out_n).read() == text_one
                res["read_sharded"] = {"gpus": gpus, "value": tn["reads"] / tn["count_s"], "unit": "reads/s",
                                       "count_s": tn["count_s"], "read_shards_per_sample": tn.get("read_shards_per_sample"),
                                       "same_table_as_one_gpu": same,
                                       "what": "the same ONE sample with --gpus N --read-shards N: batches dealt round the "
                                               "devices, sgc_reduce_counts sums the shard vectors (peer copies: the CLI asks "
                                               "for NCCL only for inputs of 8 GiB or more, its start-up takes seconds).  A "
                                               "correctness leg: a 16 M-read gzip file is host-bound on one GPU already"}
                assert same, "CLI --gpus N table differs from --gpus 1"
        if with_oracle:
            from oracle import oracle as orc

            t0 = time.perf_counter()
            recs = orc.Records.from_path(fq)
            t_parse = time.perf_counter() - t0
            lib_recs = orc.Records.from_path(lib_path)
            olib = orc.Library.from_reader(lib_recs)
            operm = orc.Permuter.new(olib)
            t0 = time.perf_counter()
            oc = orc.Counter.new(recs, olib, operm, orc.Offset.Forward(OFFSET), None, True, n_threads=1)
            t_match = time.perf_counter() - t0
            res["cpu_port"] = {"value": n_reads / (t_parse + t_match), "unit": "reads/s", "cores": 1,
                               "gunzip_parse_s": t_parse, "match_s": t_match,
                               "note": "oracle port, one thread per sample like the reference (count.rs:117-136)"}
            counts = oc.counts_by_index()
            want = {"lib.%d" % i: int(c) for i, c in enumerate(counts) if c}
            res["parity"] = "ok" if want == table else "MISMATCH"
            assert want == table, "CLI count table differs from the oracle's"
        return res
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from sgcount_b200 import synth

    threads = cpu_threads()
    lib_arr = synth.make_library(SEED, N_GUIDES, K)
    sample_reads = min(4_000_000, 250_000 * threads)
    leg = OracleLeg(lib_arr, sample_reads, threads)
    for _ in range(args.warmup):
        leg.step()
    times = [leg.step()[0] for _ in range(args.steps)]
    total = sum(times)
    value = sample_reads * args.steps / total
    one_n = min(sample_reads, 1_000_000)
    one_dt, _ = leg.step(threads=1, n=one_n)
    out = {
        "impl": "reference",
        "metric": "reads/sec matched per B200 (kernel & end-to-end)",
        "value": value,
        "unit": "reads/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u8",
        "data": "synthetic",
        "config": bench_config(args.gpus, args.reads_per_gpu),
        "cpu_baseline": {"value": value, "unit": "reads/s", "cores": threads, "kind": "port", "sample": leg.describe(),
                         "single_thread": {"value": one_n / one_dt, "unit": "reads/s", "cores": 1,
                                           "note": "what the stock reference can use for ONE sample: its only "
                                                   "parallel construct is over samples (count.rs:117-136)"}},
        "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reason_bits = 0
        self.max_mhz = None
        self.active = threading.Event()
        self.stop_flag = False
        self.ok = False
        self.pci = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if visible:
                ids = [v for v in visible.split(",") if v.strip() != ""]
                if index < len(ids) and ids[index].strip().isdigit():
                    phys = int(ids[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            try:
                bus = pynvml.nvmlDeviceGetPciInfo(self.h).busId
                self.pci = (bus.decode() if isinstance(bus, bytes) else bus).lower()
            except Exception:
                self.pci = None
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        try:  # the first queries of a process are slow: take them before anything is timed
            for _ in range(3):
                self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            pass
        while not self.stop_flag:
            if self.active.is_set():
                try:
                    mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                    try:
                        bits = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        bits = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.samples.append(mhz)
                    self.reason_bits |= int(bits)
                except Exception:
                    pass
                time.sleep(0.0005)  # an NVML query takes a fraction of a millisecond: sample back to back
            else:
                time.sleep(0.002)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        reasons = [name for bit, name in self.REASONS.items() if self.reason_bits & bit]
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(reasons),
                "samples": len(self.samples)}


BAD_REASONS = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


# ---------------------------------------------------------------------------------------------
# placement: which device a rank uses and where its pinned buffers live
# ---------------------------------------------------------------------------------------------
def pick_device(local: int, world: int, visible: int) -> int:
    """With fewer ranks than visible devices the ranks are spread over the box (0, 2, 4, 6 for four
    ranks of eight) so that neighbouring devices, which share a PCIe switch and a socket's host
    links, are not the ones copying at the same time."""
    if world < visible and visible % world == 0:
        return local * (visible // world)
    return local


def bind_to_device_numa_node(pci: str):
    """Pins this process (and so its first-touch pinned allocations) to the CPUs of the NUMA node
    the device hangs off, when the cpuset allows it.  Returns a description for the JSON line."""
    info = {"pci": pci, "numa_node": None, "bound_cpus": None}
    try:
        if not pci:
            return info
        dev = pci[-12:] if len(pci) > 12 else pci  # sysfs uses a 4-digit domain
        node = int(open(f"/sys/bus/pci/devices/{dev}/numa_node").read().strip())
        info["numa_node"] = node
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if len(allowed) >= 2:
            os.sched_setaffinity(0, allowed)
            info["bound_cpus"] = len(allowed)
    except Exception as e:  # no sysfs entry, no permission: run unbound
        info["error"] = str(e)[:80]
    return info


# ---------------------------------------------------------------------------------------------
# BASELINE configs 3-5 at full size
# ---------------------------------------------------------------------------------------------
def plan_units(cfg, world):
    """(sample position, first read, n reads, rank) of every shard: whole samples are dealt round
    the ranks; a sample with several shards has its shards dealt round the ranks."""
    units = []
    n_shards = cfg["shards_per_sample"]
    # more ranks than shards (config 3's four samples on eight GPUs): cut every sample further, so
    # that no rank idles — read shards of a sample are summed like config 5's
    while len(cfg["samples"]) * n_shards < world and cfg["reads_per_sample"] % (2 * n_shards * 32) == 0:
        n_shards *= 2
    per = cfg["reads_per_sample"] // n_shards
    assert per * n_shards == cfg["reads_per_sample"] and per % 32 == 0  # whole tiles, 16-byte aligned
    for si in range(len(cfg["samples"])):
        for sh in range(n_shards):
            slot = si * n_shards + sh
            units.append((si, sh * per, per, slot % world))
    return units


def run_full_config(name, cfg, ctx, reps, with_parity):
    """Counts one BASELINE config at full size from HBM.  Returns rank 0's dict (None elsewhere)."""
    import torch
    import torch.distributed as dist

    import sgcount_b200 as sg
    from sgcount_b200 import _cabi, synth

    world, rank, dev, local_dev = ctx["world"], ctx["rank"], ctx["dev"], ctx["device_index"]
    stream = ctx["stream"]
    n_guides, seed = cfg["n_guides"], cfg["seed"]
    n_samples = len(cfg["samples"])
    scale = ctx["scale"]
    t_setup = time.perf_counter()
    lib_arr = synth.make_library(seed, n_guides, K)
    guides = [lib_arr[i].tobytes() for i in range(n_guides)]
    library = sg.Library(guides, [b"lib.%d" % i for i in range(n_guides)], device=local_dev)
    permuter = sg.Permuter.new(library)
    info = permuter.info()
    samples = [synth.Sample(seed, idx, lib_arr, READ_LEN, off, rev) for idx, rev, off in cfg["samples"]]
    units = plan_units(cfg, world)
    if scale != 1.0:  # --config-scale: smaller runs for development; the JSON says so
        units = [(si, int(first * scale) // 32 * 32, max(32, int(n * scale) // 32 * 32), r) for si, first, n, r in units]
    mine = [u for u in units if u[3] == rank]

    # this rank's shards, generated in HBM
    bufs = []
    for si, first, n, _ in mine:
        d = torch.empty(n * STRIDE + 256, dtype=torch.uint8, device=dev)
        samples[si].fill_device(first, n, d.data_ptr(), device=local_dev, stream=stream)
        bufs.append(d)
    torch.cuda.synchronize()

    # offsets: detected ONCE per sample, on its first 5000 records, by the rank that holds them
    # (offsetter.rs:192-200), then handed to every rank
    off_t = torch.zeros((n_samples, 2), dtype=torch.int64, device=dev)
    t_detect = 0.0
    for (si, first, n, _), d in zip(mine, bufs):
        if first != 0:
            continue
        head_n = min(5000, n)
        head = d[:head_n * STRIDE].cpu().numpy()
        t0 = time.perf_counter()
        o = sg.entropy_offset(library, sg.ReadBatch(head, head_n, None, STRIDE, READ_LEN), 5000)
        t_detect += time.perf_counter() - t0
        off_t[si, 0], off_t[si, 1] = int(o.reverse), int(o.index)
    if world > 1:
        dist.all_reduce(off_t)
    offs = [(bool(r), int(i)) for r, i in off_t.cpu().tolist()]
    truth = [(rev, off) for _, rev, off in cfg["samples"]]
    assert offs == truth, f"{name}: detected offsets {offs} != planted {truth}"

    def make_counters():
        out = []
        for si, _, _, _ in mine:
            st = torch.zeros(n_guides + 2, dtype=torch.int64, device=dev)
            c = sg.Counter(library, permuter, sg.Offset(*offs[si]), True, _cabi.RC_BITTRICK, stream=stream,
                           d_state=st.data_ptr())
            out.append((c, st))
        return out

    table = torch.zeros((n_samples, n_guides + 2), dtype=torch.int64, device=dev)

    def one_pass(counters, prefix=None, events=None):
        """every shard of this rank counted, the sample table assembled on every rank"""
        table.zero_()
        for j, ((si, _, n, _), d, (c, st)) in enumerate(zip(mine, bufs, counters)):
            c.reset()
            m = n if prefix is None else min(prefix, n)
            if events is not None:
                events[j][0].record()
            c.submit_device(d.data_ptr(), m * STRIDE, m, STRIDE, READ_LEN)
            if events is not None:
                events[j][1].record()
            table[si] += st
        if world > 1:
            dist.all_reduce(table)  # the one exchange: u64[n_samples x (n_guides + 2)], NCCL over NVLink

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    setup_s = time.perf_counter() - t_setup
    counters = make_counters()
    # first pass: fresh counters (the skew plan of every counter is made here) and cold tables
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    one_pass(counters)
    b.record()
    barrier()
    first_ms = max_over_ranks(a.elapsed_time(b))
    events = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in mine] for _ in range(reps)]
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for r in range(reps):
        one_pass(counters, events=events[r])
    b.record()
    barrier()
    step_ms = max_over_ranks(a.elapsed_time(b)) / reps
    kernel_ms_local = statistics.mean(sum(x.elapsed_time(y) for x, y in ev) for ev in events) if mine else 0.0
    kernel_ms = max_over_ranks(kernel_ms_local)
    launches = sum(c.launch_info().launches_total for c, _ in counters)
    plan = [(c.launch_info().replicas, c.launch_info().hot_guides) for c, _ in counters]
    full = table.cpu().numpy().astype(np.uint64)
    total_reads = sum(u[2] for u in units)
    assert int(full[:, -2].sum()) == total_reads, (name, int(full[:, -2].sum()), total_reads)
    per_sample = [sum(u[2] for u in units if u[0] == si) for si in range(n_samples)]
    assert [int(x) for x in full[:, -2]] == per_sample
    assert all(int(full[si, :-2].sum()) == int(full[si, -1]) for si in range(n_samples))

    parity = None
    if with_parity:
        pc = make_counters()
        one_pass(pc, prefix=PARITY_PREFIX)
        torch.cuda.synchronize()
        got = table.cpu().numpy().astype(np.uint64)
        del pc
        if rank == 0:
            from oracle import oracle as orc

            lib_recs = orc.Records.from_bytes(library_fasta(lib_arr))
            olib = orc.Library.from_reader(lib_recs)
            operm = orc.Permuter.new(olib)
            want = np.zeros_like(got)
            threads = cpu_threads()
            for si, first, n, _ in units:  # EVERY rank's prefixes, regenerated on the host
                m = min(PARITY_PREFIX, n)
                lines = samples[si].fill_host(first, m)
                recs = orc.Records.from_lines(lines, np.arange(0, lines.nbytes + 1, STRIDE, dtype=np.uint64))
                if first == 0:  # the detector's answer too
                    od = orc.entropy_offset(lib_recs, recs, 5000)
                    assert (od.reverse, od.index) == offs[si], (name, si, od, offs[si])
                oc = orc.Counter.new(recs, olib, operm, orc.Offset(*offs[si]), None, True, n_threads=threads)
                want[si, :-2] += oc.counts_by_index()
                want[si, -2] += oc.total_reads()
                want[si, -1] += oc.matched_reads()
            parity = "ok" if np.array_equal(got, want) else "MISMATCH"
            if parity != "ok":  # reported in the line (and loudly here); the other configs still run
                print(f"[bench] {name}: GPU table differs from the oracle on the shard prefixes", file=sys.stderr, flush=True)

    out = None
    if rank == 0:
        peak, _ = measured_peak()
        my_bytes = sum(u[2] for u in mine) * STRIDE
        out = {
            "what": cfg["what"],
            "reads": total_reads,
            "samples": n_samples,
            "shards": len(units),
            "shards_on_rank0": len(mine),
            "n_guides": n_guides,
            "table_bytes": int(info.table_bytes),
            "scaling": "strong" if world > 1 else "1 GPU",
            "ms": step_ms,
            "kernel_ms_max_rank": kernel_ms,
            "first_pass_ms": first_ms,
            "value": total_reads / (step_ms * 1e-3),
            "unit": "reads/s",
            "frac": (my_bytes / (kernel_ms_local * 1e-3) / 1e9 / peak) if kernel_ms_local else None,
            "frac_note": "rank 0's shards: algorithmic bytes / summed kernel time / measured HBM peak",
            "offsets_detected": [("Reverse(%d)" if r else "Forward(%d)") % i for r, i in offs],
            "offset_detect_ms": 1e3 * t_detect,
            "skew_plan": sorted(set(plan)),
            "launches": int(launches),
            "matched_fraction": float(full[:, -1].sum()) / max(total_reads, 1),
            "parity": parity,
            "parity_prefix_reads_per_shard": PARITY_PREFIX if with_parity else 0,
            "setup_s": setup_s,
        }
        if scale != 1.0:
            out["scaled_to"] = scale
    del counters, bufs, table
    torch.cuda.empty_cache()
    return out


def run_fixture_config(ctx):
    """config 1: example/library.fasta.gz + example/sequence.fastq.gz through the public API, auto
    offset, checked against the committed golden table (tests/golden/example/expected.json)."""
    import sgcount_b200 as sg

    ex = os.path.join(ROOT, "tests", "golden", "example")
    expected = json.load(open(os.path.join(ex, "expected.json")))["fixtures"]["sequence"]
    t0 = time.perf_counter()
    library = sg.Library.from_reader(sg.read_fastx(os.path.join(ex, "library.fasta.gz")), device=ctx["device_index"])
    permuter = sg.Permuter.new(library)
    t1 = time.perf_counter()
    reads = sg.read_fastx(os.path.join(ex, "sequence.fastq.gz"))
    t2 = time.perf_counter()
    times = []
    for _ in range(5):
        t = time.perf_counter()
        offset = sg.entropy_offset(library, reads, 5000)
        counter = sg.Counter.new(reads, library, permuter, offset, library.size(), True)
        counts, total, matched = counter.finish()
        times.append(time.perf_counter() - t)
    ok = (counts.tolist() == expected["counts"] and total == expected["total_reads"]
          and matched == expected["matched_reads"] and (offset.reverse, offset.index) == (False, 5))
    assert ok, "config 1 differs from the golden table"
    best = min(times)
    return {"what": "config1: example/library.fasta.gz (100 guides) + example/sequence.fastq.gz (1000 x 80 bp), auto offset, "
                    "host buffers -> offset detection -> count -> table (latency bound: 1000 reads)",
            "reads": int(total), "offset": repr(offset), "ms": 1e3 * best, "value": total / best, "unit": "reads/s",
            "table_build_ms": 1e3 * (t1 - t0), "parse_ms": 1e3 * (t2 - t1), "parity": "ok (golden table)"}


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    import sgcount_b200 as sg
    from sgcount_b200 import _cabi, shard, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1")
    visible = torch.cuda.device_count()
    local_dev = pick_device(local, world, visible)
    sampler = ClockSampler(local_dev)
    all_cpus = os.sched_getaffinity(0)
    placement = bind_to_device_numa_node(sampler.pci)  # before any pinned allocation
    placement.update({"local_rank": local, "device": local_dev, "visible_devices": visible})
    torch.cuda.set_device(local_dev)
    dev = torch.device("cuda", local_dev)
    # Everything timed runs on ONE explicit (non-default) stream: the counter's kernels are
    # launched on it through the C ABI and the torch events / NCCL collectives are recorded on
    # it, so the CUDA events bracket exactly the launches they are meant to time.
    work_stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(work_stream)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n_reads = args.reads_per_gpu
    stride = STRIDE
    n_bytes = n_reads * stride

    # library + unified one-mismatch table on this GPU (replicated on every rank)
    lib_arr = synth.make_library(SEED, N_GUIDES, K)
    guides = [lib_arr[i].tobytes() for i in range(N_GUIDES)]
    library = sg.Library(guides, [b"lib.%d" % i for i in range(N_GUIDES)], device=local_dev)
    permuter = sg.Permuter.new(library)
    info = permuter.info()

    # this rank's shard of sample 0, generated in HBM
    sample = synth.Sample(SEED, 0, lib_arr, READ_LEN, OFFSET, False)
    d_lines = torch.empty(n_bytes + 256, dtype=torch.uint8, device=dev)
    first = rank * n_reads
    sample.fill_device(first, n_reads, d_lines.data_ptr(), device=local_dev, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()

    stream = work_stream.cuda_stream
    assert stream != 0 and torch.cuda.current_stream().cuda_stream == stream
    # Two counters on two state vectors: with N > 1 the all-reduce of step i runs on a second
    # stream while the kernel of step i+1 counts into the other vector, the way consecutive
    # samples of a real run overlap (sample i's reduce under sample i+1's counting).  Every
    # step's kernel AND reduce complete inside the timed region.
    n_buf = 2 if world > 1 else 1
    states = [torch.zeros(N_GUIDES + 2, dtype=torch.int64, device=dev) for _ in range(n_buf)]
    counters = [sg.Counter(library, permuter, sg.Offset.Forward(OFFSET), True, _cabi.RC_BITTRICK, stream=stream,
                           d_state=st.data_ptr()) for st in states]
    state, counter = states[0], counters[0]
    comm_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    reduce_done = [None] * n_buf

    def kernel_step(i, k_events=None):
        b = i % n_buf
        c, st = counters[b], states[b]
        if reduce_done[b] is not None:
            work_stream.wait_event(reduce_done[b])  # the vector's previous all-reduce has finished
        c.reset()
        if k_events is not None:
            k_events[0].record()
        c.submit_device(d_lines.data_ptr(), n_bytes, n_reads, stride, READ_LEN)
        if k_events is not None:
            k_events[1].record()
        if world > 1:
            counted = torch.cuda.Event()
            counted.record(work_stream)
            with torch.cuda.stream(comm_stream):
                comm_stream.wait_event(counted)
                shard.reduce_counts(st)  # NCCL all-reduce: the only state that crosses GPUs
                reduce_done[b] = torch.cuda.Event()
                reduce_done[b].record(comm_stream)

    def join_reduces():
        for ev in reduce_done:
            if ev is not None:
                work_stream.wait_event(ev)

    sampler.start()

    def timed_kernel_arm():
        for i in range(args.warmup):
            kernel_step(i)
        join_reduces()
        barrier()
        launches0 = sum(c.launch_info().launches_total for c in counters)
        k_events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.active.set()
        start.record()
        for i in range(args.steps):
            kernel_step(i, k_events[i])
        join_reduces()
        end.record()
        barrier()
        sampler.active.clear()
        total_ms = max_over_ranks(start.elapsed_time(end))
        kernel_ms = statistics.mean(a.elapsed_time(b) for a, b in k_events)
        launches = sum(c.launch_info().launches_total for c in counters) - launches0
        return total_ms, kernel_ms, launches

    total_ms, kernel_ms, launches = timed_kernel_arm()
    if set(sampler.summary()["reasons"]) & BAD_REASONS:  # rejected: measure once more
        sampler.samples.clear()
        sampler.reason_bits = 0
        total_ms, kernel_ms, launches = timed_kernel_arm()
    clocks_kernel = sampler.summary()
    clocks_kernel["window"] = "timed region"
    if clocks_kernel["samples"] < 5:
        # K steps of ~1 ms are over before NVML answers a handful of queries: sample the SAME launches,
        # back to back for a quarter of a second, right after the timed region (not part of `value`)
        sampler.active.set()
        t_end = time.perf_counter() + 0.25
        i = 0
        while time.perf_counter() < t_end:
            for _ in range(20):
                kernel_step(i)
                i += 1
            join_reduces()
            torch.cuda.synchronize()
        barrier()
        sampler.active.clear()
        clocks_kernel = sampler.summary()
        clocks_kernel["window"] = "timed region + 0.25 s of the same launches right after it"
        kernel_step(args.steps - 1)  # leave the last timed step's table in its state vector
        join_reduces()
        torch.cuda.synchronize()

    last = (args.steps - 1) % n_buf
    state, counter = states[last], counters[last]
    counts_last, total_last, matched_last = counter.finish()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, counts_last, total_last, matched_last)
    value = world * n_reads * args.steps / (total_ms * 1e-3)
    headline_plan = (counter.launch_info().replicas, counter.launch_info().hot_guides)

    # ---- parity of THIS run at every N: each rank counts a prefix of its shard into a second
    # vector, the vectors are all-reduced, rank 0 asks the oracle about the same N prefixes ----
    prefix = min(PARITY_PREFIX, n_reads)
    p_state = torch.zeros(N_GUIDES + 2, dtype=torch.int64, device=dev)
    p_counter = sg.Counter(library, permuter, sg.Offset.Forward(OFFSET), True, _cabi.RC_BITTRICK, stream=stream,
                           d_state=p_state.data_ptr())
    p_counter.submit_device(d_lines.data_ptr(), prefix * stride, prefix, stride, READ_LEN)
    if world > 1:
        shard.reduce_counts(p_state)
    p_counts, p_total, p_matched = p_counter.finish()
    del p_counter

    # ---- skew: a tenth of the resident reads rewritten to carry ONE guide.  The reference's fold
    # (counter.rs:232-235) costs the same whatever the abundances; here the counter's automatic plan
    # has to make it so (rank 0 reports; every rank does the same work) -----------------------------
    def timed_launches(c, n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            c.submit_device(d_lines.data_ptr(), n_bytes, n_reads, stride, READ_LEN)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    rows = d_lines[:n_bytes].view(n_reads, stride)
    hot_row = rows[0].clone()
    hot_row[OFFSET:OFFSET + K] = torch.from_numpy(lib_arr[12345].copy()).to(dev)
    mask = torch.rand(n_reads, device=dev) < 0.1
    rows[mask] = hot_row
    del mask
    torch.cuda.synchronize()
    sk = sg.Counter(library, permuter, sg.Offset.Forward(OFFSET), True, _cabi.RC_BITTRICK, stream=stream)
    sk_first = timed_launches(sk, 1)  # carries the plan: sample launch, top guides, one synchronisation
    sk_ms = timed_launches(sk, 5)
    sk_info = sk.launch_info()
    sk_counts = sk.finish()[0]
    plain = sg.Counter(library, permuter, sg.Offset.Forward(OFFSET), True, _cabi.RC_BITTRICK, stream=stream)
    plain.set_replicas(1)
    plain_ms = timed_launches(plain, 2)
    same_skew = bool(np.array_equal(plain.finish()[0] * 3, sk_counts))
    assert same_skew, "the skew plan changed the counts"
    skew = {"p_top": 0.1, "ms": sk_ms, "ms_uniform": kernel_ms, "ratio": sk_ms / kernel_ms, "first_launch_ms": sk_first,
            "replicas": int(sk_info.replicas), "hot_guides": int(sk_info.hot_guides), "ms_without_plan": plain_ms,
            "top_share": float(sk_counts.max()) / float(max(int(sk_counts.sum()), 1)), "same_counts": same_skew,
            "what": "10 % of the 50 M resident reads rewritten to carry one guide; default counter (automatic plan) "
                    "against the uniform sample's kernel time and against the same counter with the plan switched off"}
    del sk, plain, rows, hot_row
    sample.fill_device(first, n_reads, d_lines.data_ptr(), device=local_dev, stream=stream)
    torch.cuda.synchronize()

    # ---- end to end: pinned host lines -> sgc_counter_submit -> counts on the host -------------
    lib = _cabi.load()
    host_ptr = ctypes.c_void_p()
    _cabi.check(lib.sgc_host_alloc(ctypes.byref(host_ptr), n_bytes))
    sample.fill_host_ptr(first, n_reads, host_ptr.value)
    host_lines = np.ctypeslib.as_array(ctypes.cast(host_ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(n_bytes,))
    batch = sg.ReadBatch(host_lines, n_reads, None, stride, READ_LEN)
    e2e_counter = sg.Counter(library, permuter, sg.Offset.Forward(OFFSET), True, _cabi.RC_BITTRICK, stream=stream,
                             d_state=state.data_ptr())
    e2e_steps = max(1, min(args.steps, args.e2e_steps))

    # the ceiling of this arm: a plain pinned host->device copy of 1 GiB of the same buffer, every
    # rank at the same time (what the links and the host memory give N concurrent copies)
    probe_bytes = min(n_bytes, 1 << 30)
    h_probe = torch.from_numpy(host_lines[:probe_bytes])
    assert h_probe.is_pinned(), "the probe must copy from page-locked memory"
    d_probe = d_lines[:probe_bytes]
    pcie_gbs = []
    for it in range(4):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        d_probe.copy_(h_probe, non_blocking=True)  # cudaMemcpyAsync on the work stream: the source is pinned
        b.record()
        torch.cuda.synchronize()
        if it:
            pcie_gbs.append(probe_bytes / (a.elapsed_time(b) * 1e-3) / 1e9)
    del h_probe
    pcie_peak_local = max(pcie_gbs)
    pcie_peak_min = -max_over_ranks(-pcie_peak_local)
    # the probe overwrote the head of d_lines: regenerate it (the configs below do not use it, the
    # parity prefix was taken above)
    sample.fill_device(first, n_reads, d_lines.data_ptr(), device=local_dev, stream=stream)
    torch.cuda.synchronize()

    def e2e_step():
        e2e_counter.reset()
        e2e_counter.submit(batch)
        if world > 1:
            shard.reduce_counts(state)
        return e2e_counter.finish()

    for _ in range(min(args.warmup, 3)):
        e2e_step()
    barrier()
    sampler.samples.clear()
    sampler.active.set()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_result = e2e_step()
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    sampler.active.clear()
    clocks_e2e = sampler.summary()
    sampler.stop_flag = True
    e2e_value = world * n_reads * e2e_steps / e2e_s

    # ---- the same with SPAN records: a host that frames its own records (the CLI's ingest does)
    # sends the guide window and one byte either side, 24 bytes per read instead of 76 ----------
    span_ptr = ctypes.c_void_p()
    s_start, s_len, s_off = sg.span_geometry(K, READ_LEN, sg.Offset.Forward(OFFSET), True)
    s_stride = (s_len + 7) & ~7
    _cabi.check(lib.sgc_host_alloc(ctypes.byref(span_ptr), n_reads * s_stride))
    span_host = np.ctypeslib.as_array(ctypes.cast(span_ptr, ctypes.POINTER(ctypes.c_uint8)), shape=(n_reads * s_stride,))
    span_batch, _ = sg.span_batch(batch, K, sg.Offset.Forward(OFFSET), True, out=span_host)  # cut on the host, not timed
    span_counter = sg.Counter(library, permuter, s_off, True, _cabi.RC_BITTRICK, stream=stream, d_state=state.data_ptr())

    def span_step():
        span_counter.reset()
        span_counter.submit(span_batch)
        if world > 1:
            shard.reduce_counts(state)
        return span_counter.finish()

    for _ in range(min(args.warmup, 3)):
        span_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        span_result = span_step()
    barrier()
    span_s = max_over_ranks(time.perf_counter() - t0)
    span_value = world * n_reads * e2e_steps / span_s
    span_kernel = span_counter.launch_info().kernel
    del e2e_counter, span_counter
    _cabi.check(lib.sgc_host_free(host_ptr))
    _cabi.check(lib.sgc_host_free(span_ptr))
    os.sched_setaffinity(0, all_cpus)  # the CPU legs below get every core of the box again

    # the two arms must have produced the same table
    same = bool(np.array_equal(e2e_result[0], counts_last)) and e2e_result[1:] == (total_last, matched_last)
    assert total_last == world * n_reads, (total_last, world * n_reads)
    assert same, "kernel-only and end-to-end arms disagree"
    same_spans = bool(np.array_equal(span_result[0], counts_last)) and span_result[1:] == (total_last, matched_last)
    assert same_spans, "span records and whole lines disagree"
    placements = [placement]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, placement)
        placements = gathered

    out = None
    if rank == 0:
        peak, peak_src = measured_peak()
        algo_bytes = n_reads * stride
        achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get("count_stream_kernel_dram_bytes_per_launch")
            except Exception:
                traffic = None
        e2e_gbs = n_bytes * e2e_steps / e2e_s / 1e9  # per rank
        out = {
            "metric": "reads/sec matched per B200 (kernel & end-to-end)",
            "value": value,
            "unit": "reads/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "u8",
            "data": "synthetic",
            "config": bench_config(world, n_reads),
            "details": {
                "table_bytes": int(info.table_bytes),
                "n_variants": int(info.n_variants),
                "n_ambiguous": int(info.n_ambiguous),
                "table_build_ms": float(info.build_ms),
                "matched_fraction": matched_last / max(total_last, 1),
                "skew_plan": {"replicas": headline_plan[0], "hot_guides": headline_plan[1]},
                "placement": placements,
            },
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": n_bytes,
                    "d2h_bytes_per_step": (N_GUIDES + 2) * 8, "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
                    "roofline": {"bound": "pcie", "achieved": e2e_gbs, "peak": pcie_peak_min, "unit": "GB/s",
                                 "frac": e2e_gbs / pcie_peak_min,
                                 "note": f"per rank: H2D bytes / step time; peak = a plain pinned cudaMemcpyAsync of "
                                         f"{probe_bytes >> 20} MiB measured in this run with all {world} rank(s) copying at "
                                         "once (slowest rank).  The arm only gets faster by sending fewer bytes per read."}},
            "e2e_spans": {"value": span_value, "unit": "reads/s", "h2d_bytes_per_step": n_reads * s_stride,
                          "d2h_bytes_per_step": (N_GUIDES + 2) * 8, "steps": e2e_steps,
                          "ms_per_step": 1e3 * span_s / e2e_steps, "bytes_per_read": s_stride, "span": [s_start, s_len],
                          "same_table": same_spans, "kernel": "streaming" if span_kernel == 0 else "lines",
                          "roofline": {"bound": "pcie", "achieved": n_reads * s_stride * e2e_steps / span_s / 1e9,
                                       "peak": pcie_peak_min, "unit": "GB/s",
                                       "frac": n_reads * s_stride * e2e_steps / span_s / 1e9 / pcie_peak_min},
                          "what": "NOT the headline e2e (which copies whole 76-byte sequence lines): the host hands "
                                  "sgc_counter_submit pinned SPAN records, bytes [offset-1, offset+k+1) of every read "
                                  f"in {s_stride}-byte records (sgc_span_geometry), as the CLI's ingest frames them for "
                                  "fixed-length reads; cutting them out of the lines is host framing work, not timed here"},
            "skew": skew,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "kernel_ms": kernel_ms,
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "note": "kernel = count_stream_kernel (the only count launch of a step: 50 M reads are whole 32-read tiles); "
                                 "duration = CUDA events around sgc_counter_submit_device on the launching stream, mean over the timed steps; "
                                 "traffic = dram bytes of one launch from the committed ncu --set full capture (profiles/traffic.json)"},
            "clocks": {"sm_mhz": clocks_kernel["sm_mhz"], "sm_max_mhz": clocks_kernel["sm_max_mhz"],
                       "reasons": clocks_kernel["reasons"], "samples": clocks_kernel["samples"],
                       "window": clocks_kernel["window"], "e2e_sm_mhz": clocks_e2e["sm_mhz"]},
        }
        if not args.no_cpu_baseline:
            # parity of the bench's own run, at every N: the oracle over the N shard prefixes
            from oracle import oracle as orc

            threads = cpu_threads()
            lib_recs = orc.Records.from_bytes(library_fasta(lib_arr))
            olib = orc.Library.from_reader(lib_recs)
            t0 = time.perf_counter()
            operm = orc.Permuter.new(olib)
            permuter_s = time.perf_counter() - t0
            want = np.zeros(N_GUIDES + 2, dtype=np.uint64)
            for r in range(world):
                lines = sample.fill_host(r * n_reads, prefix)
                recs = orc.Records.from_lines(lines, np.arange(0, lines.nbytes + 1, stride, dtype=np.uint64))
                oc = orc.Counter.new(recs, olib, operm, orc.Offset.Forward(OFFSET), None, True, n_threads=threads)
                want[:-2] += oc.counts_by_index()
                want[-2] += oc.total_reads()
                want[-1] += oc.matched_reads()
            ok = (np.array_equal(p_counts.astype(np.uint64), want[:-2]) and p_total == int(want[-2])
                  and p_matched == int(want[-1]))
            out["parity_n"] = "ok" if ok else "MISMATCH"
            out["parity_n_note"] = (f"every rank counted the first {prefix} reads of its shard into a second vector, "
                                    f"all-reduced over {world} rank(s); the oracle counted the same {world} prefixes")
            assert ok, "GPU counts differ from the oracle on the shard prefixes"
            if world == 1:
                sample_reads = min(4_000_000, 250_000 * threads, n_reads)
                leg = OracleLeg(lib_arr, sample_reads, threads)
                dt, oc = leg.step()
                one_n = min(sample_reads, 1_000_000)
                one_dt, _ = leg.step(threads=1, n=one_n)
                out["cpu_baseline"] = {"value": sample_reads / dt, "unit": "reads/s", "cores": threads, "kind": "port",
                                       "sample": leg.describe(),
                                       "single_thread": {"value": one_n / one_dt, "unit": "reads/s", "cores": 1,
                                                         "note": "what the stock reference can use for ONE sample "
                                                                 "(count.rs:117-136 parallelises over samples only)"}}
                # parity of the cpu_baseline sample itself
                chk = sg.Counter(library, permuter, sg.Offset.Forward(OFFSET), True, _cabi.RC_BITTRICK, stream=stream)
                chk.submit_device(d_lines.data_ptr(), sample_reads * stride, sample_reads, stride, READ_LEN)
                g_counts, g_total, g_matched = chk.finish()
                ok = (np.array_equal(g_counts, oc.counts_by_index()) and g_total == oc.total_reads()
                      and g_matched == oc.matched_reads())
                out["parity"] = "ok" if ok else "MISMATCH"
                assert ok, "GPU counts differ from the oracle on the cpu_baseline sample"
            else:
                out["parity"] = out["parity_n"]
            del operm, olib

    if rank == 0:
        print(f"[bench] headline: {json.dumps(out)}", file=sys.stderr, flush=True)
    # ---- the other BASELINE configs at full size -------------------------------------------------
    del counters, states, d_lines, d_probe
    torch.cuda.empty_cache()
    wanted = [c.strip() for c in args.configs.split(",") if c.strip()]
    ctx = {"world": world, "rank": rank, "dev": dev, "device_index": local_dev, "stream": stream,
           "scale": args.config_scale}
    cfg_out = {}
    if "c1" in wanted and rank == 0:
        cfg_out["c1"] = run_fixture_config(ctx)
    for name in ("c3", "c4", "c5"):
        if name in wanted:
            res = run_full_config(name, CONFIGS[name], ctx, args.config_reps, with_parity=not args.no_cpu_baseline)
            if rank == 0:
                cfg_out[name] = res
                print(f"[bench] {name}: {json.dumps(res)}", file=sys.stderr, flush=True)
    if rank == 0:
        out["configs"] = cfg_out
        if args.fastq_reads > 0:
            out["e2e_fastq"] = fastq_leg(lib_arr, args.fastq_reads, with_oracle=(world == 1 and not args.no_cpu_baseline),
                                         gpus=world)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads-per-gpu", type=int, default=READS_PER_GPU)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="also skips every oracle parity check")
    ap.add_argument("--fastq-reads", type=int, default=16 << 20,
                    help="reads of the gzip-FASTQ end-to-end leg through the C++ host (0 = skip)")
    ap.add_argument("--configs", default="c1,c3,c4,c5", help="BASELINE configs measured besides the headline (''= none)")
    ap.add_argument("--config-reps", type=int, default=3)
    ap.add_argument("--config-scale", type=float, default=1.0,
                    help="development only: fraction of the reads of configs 3-5 (reported as scaled_to)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's per-guide counts, total and matched reads to DIR/<name>.npy "
                         "(float64; the GPU arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the GPU arm; the reference arm counts a host-dependent number of reads")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
