#!/usr/bin/env python
"""bench.py — compaction throughput of the B200 engine on BASELINE.json's metric.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    (also writes the last timed step's outputs)

A "step" is one whole compaction job over the workload (SURVEY.md 8d / BASELINE.md §3 config 2:
8-way major compaction, 100 M entries, 32-B DocKey + 256-B value, kNoCompression SSTs). With N>1
every rank compacts its own tablet of that shape (tablets are independent: no data-path
collective, weak scaling).

JSON line (one, rank 0): metric = GB/s of input bytes merged (raw key+value bytes of the input
entries, as rocksdb.raw.key.size + rocksdb.raw.value.size count them).
  value     inputs already resident in HBM, input block checksums VERIFIED (the reference default,
            rocksdb/util/options.cc:135): whole job device pipeline, wall clock between syncs.
            value_no_verify: the same without verification (informational).
  e2e       same compaction through the C ABI with HOST (pinned) input files and ONE HOST output table:
            H2D of every input file and D2H of the result inside the timed region. The compaction runs
            as --subcompactions key ranges pipelined on private streams (ybgpu_compact_files_one_table, --in-flight
            host threads, copy slots) so that H2D / kernels / D2H of different ranges overlap; every range's data
            lands at its final offset and the ONE metadata file (rebased index / filter index) is assembled while
            later ranges run — the shape DocDB's single-level universal layout (and the reference arm) writes.
            e2e.range_files = the same with one SST per range (ybgpu_compact_files);
            e2e.single_job = one job, H2D / run / D2H back to back. e2e.pcie_ceiling_gbs = concurrent
            bidirectional copies of the same pinned buffers, measured in this run.
  roofline  dominant kernel, algorithmic bytes / its CUDA-event time (see DESIGN.md); roofline.traffic is
            read from the committed ncu capture under profiles/ (traffic_source says which), not measured here.
  configs   BASELINE configs[2] (64 tablets x 4-way x 10 M: 8 tablets per GPU) and configs[3] (MVCC-heavy, the
            largest size resident on one GPU) as sub-results with their own pipeline roofline.
  cpu_baseline  the oracle (CPU restatement of the reference loop) on a bounded sample, 1 thread like the
            reference (max_subcompactions = 1), plus all_cores: the reference's pool size and all hardware
            threads running independent one-thread compactions.
  parity_check  the GPU engine compacts the cpu_baseline sample files in this run: counters, KV hash and the
            SHA-256 of both output files must equal the oracle's.
"""
import argparse
import ctypes
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEFAULT_ROWS = 100_000_000       # config 2: 100 M entries
VALUE_LEN = 256
NUM_FILES = 8
WORKLOAD = "8-way major compaction, 100M keys, 32-B DocKey / 256-B value, 1 GPU"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=DEFAULT_ROWS, help="entries per tablet (debug: smaller)")
    ap.add_argument("--sample-rows", type=int, default=6_000_000, help="entries in the CPU-baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--verify", type=int, default=1, help="verify input block checksums (reference default: on)")
    ap.add_argument("--subcompactions", type=int, default=32,
                    help="e2e arm: key-range subcompactions per job (DBOptions::max_subcompactions; 1 = one job, one output file)")
    ap.add_argument("--in-flight", type=int, default=12, help="e2e arm: subcompactions in flight (host threads / private streams)")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the BASELINE configs[2] / configs[3] sub-results")
    ap.add_argument("--c3-tablets", type=int, default=8, help="configs[2]: tablets per GPU (64 tablets / 8 GPUs)")
    ap.add_argument("--c3-rows", type=int, default=10_000_000, help="configs[2]: entries per tablet")
    ap.add_argument("--c4-rows", type=int, default=200_000_000,
                    help="configs[3] (MVCC-heavy, 20 versions/key): entries resident on one GPU (the full 1 G entries = 310 GB do not fit HBM)")
    ap.add_argument("--c5-rows-per-gpu", type=int, default=40_000_000,
                    help="configs[4] (one oversized tablet, 32-way, key-range sharded over the GPUs with NCCL): entries per GPU")
    ap.add_argument("--c5-timeout", type=float, default=240.0, help="configs[4]: give up (and still print the line) after this many seconds")
    ap.add_argument("--workload", default="config2", choices=["config2", "mvcc"],
                    help="config2 = BASELINE configs[1] (the bench line); mvcc = configs[3] shape (20 versions/key, "
                         "history cutoff drops 90 %%), scaled to --rows entries, for profiles/ only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (counters, KV-stream digest, a "
                         "fixed sample of the output files) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU engine's outputs: it needs --impl ours")
    return args


DUMP_FILE_BYTES = 2 << 20        # bytes sampled per output file: four files as float32 stay well under 64 MB
DUMP_WINDOW = 4096
DUMP_COUNTERS = ("num_input_records", "num_output_records", "num_record_drop_hidden", "num_record_drop_obsolete",
                 "num_record_drop_feed", "total_input_raw_key_bytes", "total_input_raw_value_bytes",
                 "total_output_raw_key_bytes", "total_output_raw_value_bytes", "num_output_data_blocks",
                 "output_data_file_size", "output_meta_file_size")


def dump_counters(dumps, prefix, stats):
    dumps[prefix + "_counters"] = np.array([stats[k] for k in DUMP_COUNTERS], dtype=np.float64)


def dump_file_sample(dumps, prefix, buf):
    """A file the caller receives, as float32 bytes: whole when it fits DUMP_FILE_BYTES, else DUMP_WINDOW-byte windows at
    seeded offsets (the same for the same file size) plus the last window (the footer); the offsets go alongside."""
    buf = np.asarray(buf, dtype=np.uint8)
    if buf.size <= DUMP_FILE_BYTES:
        dumps[prefix] = buf.astype(np.float32)
        return
    n = buf.size // DUMP_WINDOW
    picks = np.random.default_rng(0).choice(n, DUMP_FILE_BYTES // DUMP_WINDOW - 1, replace=False) * DUMP_WINDOW
    starts = np.unique(np.append(picks, buf.size - DUMP_WINDOW))
    dumps[prefix] = buf[starts[:, None] + np.arange(DUMP_WINDOW)].astype(np.float32)
    dumps[prefix + "_offsets"] = starts.astype(np.float64)


def write_dumps(out_dir, dumps):
    if sum(a.nbytes for a in dumps.values()) > 64 << 20:
        raise ValueError("output dump over 64 MB")
    if any(a.dtype not in (np.float32, np.float64) for a in dumps.values()):
        raise ValueError("output dump arrays must be float32 or float64")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in dumps.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(float(s[0])) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """--impl reference: the reference's CPU loop (oracle port; the reference tree itself cannot be
    compiled in this image) on the host cores. One compaction = one thread, as in the reference
    (rocksdb/util/options.cc:258, db/compaction.cc:593-604), on a bounded sample of the workload.
    Two informational figures ride along: many independent tablets on all cores, and the same
    compaction cut into key ranges with one thread per range (the CPU counterpart of the GPU arm's
    pipelined subcompactions)."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as o
    rows = min(args.rows, args.sample_rows)
    cfg = o.GenConfig(seed=2, num_rows=rows, cols=1, versions=1, num_files=NUM_FILES, value_len=VALUE_LEN)
    ssts = o.Sst.generate_all(cfg, o.TableOptions())
    in_bytes = sum(s.raw_bytes for s in ssts)
    params = o.CompactionParams()
    times = []
    # N GPUs compact N tablets at once (tablet-per-GPU): the CPU counterpart is N concurrent compactions, one thread
    # each (the reference cannot use more than one thread per compaction: max_subcompactions = 1,
    # rocksdb/util/options.cc:258; db/compaction.cc:593-604), each on its own copy of the sample.
    from concurrent.futures import ThreadPoolExecutor
    conc = max(1, args.gpus)
    n_out_box = [0]

    def one(_):
        r = o.compact(ssts, params, o.TableOptions(filter_policy=1), mode=o.BUILD_SST | o.NO_HASH, verify=bool(args.verify))
        n_out_box[0] = r.stats.num_output_records
        del r
    with ThreadPoolExecutor(conc) as ex:
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            list(ex.map(one, range(conc)))
            t1 = time.perf_counter()
            if i >= args.warmup:
                times.append(t1 - t0)
    n_out = n_out_box[0]
    total = sum(times)
    gbs = conc * in_bytes * args.steps / total / 1e9
    sample = "%d entries (%0.2f GB raw) of the same 8-way shape, %d output entries" % (rows, in_bytes / 1e9, n_out)
    # Informational (SURVEY 8d): what the host delivers across MANY tablets (one compaction is one thread in the
    # reference: max_subcompactions = 1, rocksdb/util/options.cc:258; universal compaction with one level never
    # forms subcompactions, db/compaction.cc:593-604) — the CPU counterpart of N GPUs each compacting its own tablet.
    try:
        many = all_cores_cpu(o, args)
    except Exception as e:   # never fail the arm because of the informational figure
        many = {"error": str(e)}
    line = {
        "impl": "reference", "metric": "compaction GB/s (input bytes merged)", "value": round(gbs, 4), "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(total / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample, "threads_per_compaction": 1, "concurrent_compactions": conc,
                   "same_config_note": "one-thread throughput is independent of the job size; the sample bounds the run time"},
        "mkeys_per_s": round(conc * rows * args.steps / total / 1e6, 3),
        "cpu_baseline": {"value": round(gbs, 4), "unit": "GB/s", "cores": conc, "kind": "port", "sample": sample},
        "e2e": {"value": round(gbs, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "all_cores": many,
    }
    emit_json_line(line)


# ------------------------------------------------------------------------------------------------
def all_cores_cpu(o, args, rows_each=1_000_000, min_seconds=4.0):
    """The host's compaction rate across MANY tablets: P concurrent one-thread compactions, P = the reference's
    compaction pool size floor(ncpu * 3.5 / 8) (docdb_rocksdb_util.cc:630-641), plus the all-hardware-threads figure.
    One PROCESS per compaction (oracle/cpu_worker.py): tablets share nothing in the reference, and threads of one
    process would contend on the allocator. All workers start their timed loop at the same wall-clock instant and
    run for min_seconds; the aggregate is the sum of the workers' own rates."""
    ncpu = os.cpu_count() or 1
    worker = os.path.join(ROOT, "oracle", "cpu_worker.py")
    out = {}

    def whole_machine():
        # the bench process may be bound to its GPU's NUMA node (ybgpu_bind_thread_to_device): the CPU figure must not be
        try:
            os.sched_setaffinity(0, range(ncpu))
            ctypes.CDLL(None, use_errno=True).syscall(238, 0, None, 0)       # set_mempolicy(MPOL_DEFAULT) on x86-64
        except Exception:
            pass
    for label, T in (("pool", max(1, int(ncpu * 3.5 / 8))), ("all_threads", ncpu)):
        start_at = time.time() + 3.0 + 0.02 * T          # interpreter start + sample generation of every worker
        procs = [subprocess.Popen([sys.executable, worker, "--rows", str(rows_each), "--seconds", str(min_seconds),
                                   "--start-at", "%.3f" % start_at, "--verify", str(int(bool(args.verify)))],
                                  stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, preexec_fn=whole_machine) for _ in range(T)]
        rate, done, late = 0.0, 0, 0
        for p_ in procs:
            txt, _ = p_.communicate(timeout=120 + 10 * min_seconds)
            try:
                r = json.loads(txt.strip().splitlines()[-1])
                rate += r["done"] * r["bytes_each"] / r["elapsed"]
                done += r["done"]
            except Exception:
                late += 1
        out[label] = {"value": round(rate / 1e9, 3), "unit": "GB/s", "processes": T,
                      "sample": "%d one-thread compactions of %d entries each in %d concurrent processes, %.0f s each%s" % (
                          done, rows_each, T, min_seconds, (", %d workers failed" % late) if late else "")}
    out["host_threads"] = ncpu
    return out


def cpu_baseline(args, pkg=None, device=0):
    """The oracle (CPU restatement of the reference loop) on a bounded sample, one thread; when `pkg` is given the GPU
    engine compacts the SAME sample files and every counter, the KV-stream hash and both output files' SHA-256 must equal
    the oracle's (parity_check)."""
    import hashlib
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as o
    rows = min(args.rows, args.sample_rows)
    cfg = o.GenConfig(seed=2, num_rows=rows, cols=1, versions=1, num_files=NUM_FILES, value_len=VALUE_LEN)
    ssts = o.Sst.generate_all(cfg, o.TableOptions())
    in_bytes = sum(s.raw_bytes for s in ssts)
    t0 = time.perf_counter()
    r = o.compact(ssts, o.CompactionParams(), o.TableOptions(filter_policy=1), mode=o.BUILD_SST | o.NO_HASH, verify=bool(args.verify))
    dt = time.perf_counter() - t0
    del r
    base = {"value": round(in_bytes / dt / 1e9, 4), "unit": "GB/s", "cores": 1, "kind": "port",
            "sample": "%d entries (%0.2f GB raw) of the same 8-way shape, %.1f s on one host thread (the reference "
                      "runs one thread per compaction; one-thread throughput does not depend on the job size)" % (rows, in_bytes / 1e9, dt),
            "mkeys_per_s": round(rows / dt / 1e6, 3)}
    parity = None
    if pkg is not None:
        try:
            exp = o.compact(ssts, o.CompactionParams(), o.TableOptions(filter_policy=1), mode=o.BUILD_SST, verify=bool(args.verify))
            job = pkg.GpuCompactionJob(device=device, verify_checksums=bool(args.verify), filter_policy=1)
            for s_ in ssts:
                job.add_input_sst(s_.meta_view(), s_.data_view())
            st = job.run()
            es = exp.stats
            counters = {
                "num_input_records": (st.num_input_records, es.num_input_records),
                "num_output_records": (st.num_output_records, es.num_output_records),
                "drop_hidden": (st.num_record_drop_hidden, es.num_dropped_hidden),
                "drop_obsolete": (st.num_record_drop_obsolete, es.num_dropped_obsolete),
                "drop_feed": (st.num_record_drop_feed, es.num_dropped_feed),
                "in_key_bytes": (st.total_input_raw_key_bytes, es.in_key_bytes), "in_val_bytes": (st.total_input_raw_value_bytes, es.in_val_bytes),
                "out_key_bytes": (st.total_output_raw_key_bytes, es.out_key_bytes), "out_val_bytes": (st.total_output_raw_value_bytes, es.out_val_bytes),
                "kv_hash": (job.digest(), es.kv_hash),
            }
            data, meta = job.fetch_output()
            ref = exp.sst()
            sha = lambda b_: hashlib.sha256(b_).hexdigest()
            files = {"data_sha256": (sha(data.tobytes()), sha(ref.data)), "meta_sha256": (sha(meta.tobytes()), sha(ref.meta))}
            bad = [k for k, (a, b_) in list(counters.items()) + list(files.items()) if a != b_]
            parity = {"entries": int(rows), "ok": not bad, "mismatch": bad, "kv_hash": "%016x" % counters["kv_hash"][0],
                      "data_sha256": files["data_sha256"][0][:16], "meta_sha256": files["meta_sha256"][0][:16],
                      "checked": sorted(list(counters) + list(files)), "against": "oracle (CPU port) on the cpu_baseline sample files"}
            job.close()
        except Exception as ex:
            parity = {"ok": False, "error": "%s: %s" % (type(ex).__name__, ex)}
    try:
        base["all_cores"] = all_cores_cpu(o, args)
    except Exception as ex:
        base["all_cores"] = {"error": str(ex)}
    return base, parity


_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly one JSON line: anything libraries print there (NCCL's version banner, torchrun
    notices) is rerouted to stderr; the JSON goes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_json_line(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def resident_arm(pkg, torch, ssts, handles, local_rank, stream_ptr, job_kw, verify, steps, warmup, barrier, world, dist, sample_clocks=False,
                 read_last=None):
    """`steps` whole jobs with the input files resident in HBM, timed between barriers (CUDA events + wall clock,
    max over ranks). Returns (total seconds, per-step stats, clocks, host ms per phase). With `read_last`, the last timed
    job is not closed inside the timed region: read_last(job) reads its outputs after that region, while the device input
    files the job reads from are still allocated, and the job is closed after it."""
    kept = []
    dev_files = []
    for s in ssts:
        v = s.data_view()
        t = torch.empty(v.size + 64, dtype=torch.uint8, device="cuda")
        t[16:16 + v.size].copy_(torch.from_numpy(v))
        dev_files.append(t)
    host_ms = {"create": 0.0, "add_inputs": 0.0, "run": 0.0, "close": 0.0}

    def step(keep=False):
        t0 = time.perf_counter()
        job = pkg.GpuCompactionJob(device=local_rank, verify_checksums=bool(verify), cuda_stream=stream_ptr, **job_kw)
        t1 = time.perf_counter()
        for t, s, (off, sz) in zip(dev_files, ssts, handles):
            job.add_input_device(t.data_ptr() + 16, s.data_view().size, off, sz)
        t2 = time.perf_counter()
        st = job.run()
        t3 = time.perf_counter()
        d = st.as_dict()
        if keep:
            kept.append(job)
        else:
            job.close()
        t4 = time.perf_counter()
        for k, v in zip(("create", "add_inputs", "run", "close"), (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
            host_ms[k] += v * 1e3
        return d

    for _ in range(warmup):
        step()
    for k in host_ms:
        host_ms[k] = 0.0
    clocks = ClockSampler(local_rank) if sample_clocks else None
    barrier()
    if clocks:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    stats = [step(keep=read_last is not None and i == steps - 1) for i in range(steps)]
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    clock_info = clocks.stop() if clocks else None
    step_s = max(wall, e0.elapsed_time(e1) / 1e3)
    tt = torch.tensor([step_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    for job in kept:
        try:
            read_last(job)
        finally:
            job.close()
    del dev_files             # only now: the jobs read their inputs in place (ybgpu_job_add_input_device)
    return float(tt.item()), stats, clock_info, {k: round(v / steps, 3) for k, v in host_ms.items()}


def pipeline_roofline(stats, in_bytes, hbm_peak, steps):
    gpu_s = sum(s["gpu_seconds"] for s in stats) / steps
    out_bytes = stats[-1]["total_output_raw_key_bytes"] + stats[-1]["total_output_raw_value_bytes"]
    ach = (in_bytes + out_bytes) / gpu_s / 1e9 if gpu_s > 0 else 0.0
    return {"algorithmic_bytes": int(in_bytes + out_bytes), "gpu_ms": round(gpu_s * 1e3, 3), "achieved": round(ach, 1),
            "peak": hbm_peak, "unit": "GB/s", "frac": round(ach / hbm_peak, 4)}


def main():
    quiet_stdout()
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    pkg = importlib.import_module("yugabyte-db_b200")
    if not torch.cuda.is_available() or pkg.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the compaction engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    # Host placement first: every buffer this rank allocates below (generated input files, pinned output arenas) and
    # every thread it starts must sit on the NUMA node of its GPU, or the e2e arm pays the inter-socket link
    # (profiles/h2d_d2h_ceiling.py measures the difference).
    numa_node, numa_cpus = pkg.bind_thread_to_device(local_rank)
    if world > 1:
        # keep stdout to the one JSON line: NCCL prints its version banner to stdout at NCCL_DEBUG=VERSION
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        if rank == 0:
            sys.stderr.write("[bench] NCCL communicator: %d ranks, backend %s, local_rank %d, NCCL %s\n" % (
                dist.get_world_size(), dist.get_backend(), local_rank, ".".join(map(str, torch.cuda.nccl.version()))))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peaks, peak_kind = measured_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))

    # ---- inputs: this rank's tablet (distinct key range per rank) ----
    versions = 20 if args.workload == "mvcc" else 1
    nrows = args.rows // versions
    cfg = pkg.GenConfig(seed=2 + rank, num_rows=nrows, cols=1, versions=versions, num_files=NUM_FILES, value_len=VALUE_LEN,
                        row_offset=rank * nrows, hash_rows_total=nrows * world)
    # DocDB tables carry the DocKeyV3 fixed-size bloom filter (docdb_rocksdb_util.cc:761-763): both arms build it
    job_kw = {"filter_policy": 1}
    if args.workload == "mvcc":
        # versions 0..18 are at or below the cutoff (only the newest of them survives), version 19 is above
        job_kw["cutoff_ht"] = ((cfg.base_micros + 18 * 1000 + 500) << 12)
    t0 = time.perf_counter()
    ssts = pkg.generate_ssts(cfg, max_threads=NUM_FILES)
    gen_s = time.perf_counter() - t0
    in_bytes = sum(s.raw_bytes for s in ssts)
    n_entries = sum(s.num_entries for s in ssts)
    file_bytes = sum(s.data_view().size for s in ssts)

    # block handles from each file's own index (host, once; not part of the hot path)
    handles = [read_handles(pkg, s) for s in ssts]
    stream_ptr = torch.cuda.current_stream().cuda_stream

    # ---- HBM-resident arm: checksum verification ON like the reference (verify_checksums_in_compaction = true,
    # rocksdb/util/options.cc:135, db/version_set.cc:3791-3792); the no-verify figure rides along ----
    dump = args.dump_outputs and rank == 0
    dumps = {}
    dump_info = {"dir": args.dump_outputs,
                 "note": "the last timed resident step's job.close() ran after the timed region (its outputs were read "
                         "first): compare timings with runs without --dump-outputs only with that in mind"}

    def read_resident(job):
        d = job.digest()
        dumps["value_kv_digest"] = np.array([d >> 32, d & 0xffffffff], dtype=np.float64)      # two exact halves
        data, meta = job.fetch_output()
        free, total = torch.cuda.mem_get_info()          # inputs, job buffers and the digest's KV stream all live here
        dump_info["device_gb_in_use_while_reading"] = round((total - free) / 1e9, 1)
        dump_counters(dumps, "value", job.stats().as_dict())         # output file sizes are known once fetched
        dump_file_sample(dumps, "value_data", data)
        dump_file_sample(dumps, "value_meta", meta)
    total_s, stats, clock_info, host_ms = resident_arm(pkg, torch, ssts, handles, local_rank, stream_ptr, job_kw, args.verify,
                                                       args.steps, args.warmup, barrier, world, dist, sample_clocks=True,
                                                       read_last=read_resident if dump else None)
    nv_steps = max(1, min(args.steps, 5))
    nv_s, nv_stats, _, _ = resident_arm(pkg, torch, ssts, handles, local_rank, stream_ptr, job_kw, 0, nv_steps, 1, barrier, world, dist)
    launches = sum(s["gpu_kernel_launches"] for s in stats)
    out_bytes = stats[-1]["total_output_raw_key_bytes"] + stats[-1]["total_output_raw_value_bytes"]
    phases = [sum(s["phase_seconds"][i] for s in stats) / args.steps for i in range(5)]
    enc_kernel_s = sum(s["phase_seconds"][5] for s in stats) / args.steps      # block assembler alone (CUDA events around its launch)
    torch.cuda.empty_cache()

    # ---- e2e arm: host (pinned) files in, host files out ----
    e2e = None
    if not args.no_e2e:
        cudart = torch.cuda.cudart()
        pinned = []
        for s in ssts:
            v = s.data_view()
            rc = cudart.cudaHostRegister(v.ctypes.data, v.size, 0)
            pinned.append((v, int(rc) == 0))

        # pinned host buffers for the output files, reused by every step
        out_data = torch.empty(file_bytes + (64 << 20), dtype=torch.uint8, pin_memory=True).numpy()
        out_meta = torch.empty(max(64 << 20, file_bytes // 100), dtype=torch.uint8, pin_memory=True).numpy()

        # what the link itself gives this rank: both directions at once, 32 MB chunks, the bench's own buffers
        def pcie_ceiling():
            n = min(int(file_bytes), 4 << 30) & ~0xfffff
            n = min(n, int(pinned[0][0].size)) & ~0xfffff
            src = torch.from_numpy(pinned[0][0])[:n]
            dst = torch.from_numpy(out_data)[:n]
            din = torch.empty(n, dtype=torch.uint8, device="cuda")
            dout = torch.empty(n, dtype=torch.uint8, device="cuda")
            s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
            res = {}
            for mode in ("h2d", "d2h", "both"):
                barrier()
                t0 = time.perf_counter()
                for _ in range(2):
                    for off in range(0, n, 32 << 20):
                        if mode != "d2h":
                            with torch.cuda.stream(s1):
                                din[off:off + (32 << 20)].copy_(src[off:off + (32 << 20)], non_blocking=True)
                        if mode != "h2d":
                            with torch.cuda.stream(s2):
                                dst[off:off + (32 << 20)].copy_(dout[off:off + (32 << 20)], non_blocking=True)
                s1.synchronize(); s2.synchronize()
                dt = time.perf_counter() - t0
                te = torch.tensor([dt], dtype=torch.float64, device="cuda")
                if world > 1:
                    dist.all_reduce(te, op=dist.ReduceOp.MAX)
                res[mode] = round(world * 2 * n / float(te.item()) / 1e9, 1)      # per direction, aggregate over ranks
            return res
        try:
            ceiling = pcie_ceiling()
        except Exception as ex:
            ceiling = {"error": "%s: %s" % (type(ex).__name__, ex)}
        torch.cuda.empty_cache()

        e2e_ms = {"add_inputs_h2d": 0.0, "run": 0.0, "fetch_output_d2h": 0.0, "close": 0.0}

        def step_e2e():
            t0 = time.perf_counter()
            job = pkg.GpuCompactionJob(device=local_rank, verify_checksums=bool(args.verify), cuda_stream=stream_ptr, **job_kw)
            for s, (off, sz) in zip(ssts, handles):
                job.add_input(s.data_view(), off, sz)
            t1 = time.perf_counter()
            job.run()
            t2 = time.perf_counter()
            data, meta = job.fetch_output(out_data, out_meta)
            t3 = time.perf_counter()
            st = job.stats().as_dict()
            job.close()
            t4 = time.perf_counter()
            for k, v in zip(e2e_ms, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                e2e_ms[k] += v * 1e3
            return st, data.size + meta.size

        def timed(step_fn, steps):
            for _ in range(min(args.warmup, 2) if args.rows >= 50_000_000 else args.warmup):
                step_fn()
            for k in e2e_ms:
                e2e_ms[k] = 0.0
            barrier()
            t0 = time.perf_counter()
            res = [step_fn() for _ in range(steps)]
            barrier()
            dt = time.perf_counter() - t0
            te = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return float(te.item()), res

        info_steps = max(1, min(args.steps, 5))          # the two informational modes; the headline runs args.steps
        e2e_s, res = timed(step_e2e, info_steps)
        single = {"value": round(in_bytes * world * info_steps / e2e_s / 1e9, 4), "unit": "GB/s", "steps": info_steps,
                  "h2d_bytes_per_step": int(res[-1][0]["h2d_bytes"]), "d2h_bytes_per_step": int(res[-1][0]["d2h_bytes"]),
                  "ms_per_step": round(e2e_s / info_steps * 1e3, 2), "output_file_bytes": int(res[-1][1]),
                  "host_ms_per_step": {k: round(v / info_steps, 2) for k, v in e2e_ms.items()},
                  "mode": "one ybgpu_job: H2D of all inputs, run, D2H of the one output file, back to back"}

        def verify_outputs(file_list, stride=257):
            # host-side CRC32C check of every stride-th output data block (outside the timed regions): the full-size
            # outputs cannot be compared with the oracle, but a wrong or torn device->host copy cannot pass this
            try:
                checked = bad = 0
                for meta_v, data_v in file_list:
                    c, b_ = pkg.sst_verify_blocks(meta_v, data_v, stride)
                    checked += c
                    bad += b_
                return {"blocks_checked": int(checked), "bad_blocks": int(bad), "stride": stride}
            except Exception as ex:
                return {"error": "%s: %s" % (type(ex).__name__, ex)}

        try:
            dlen = int(res[-1][0]["output_data_file_size"])
            mlen = int(res[-1][0]["output_meta_file_size"])
            single["output_check"] = verify_outputs([(out_meta[:mlen], out_data[:dlen])])
        except Exception as ex:
            single["output_check"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        e2e = dict(single, pinned_inputs=all(ok for _, ok in pinned), verify_checksums=bool(args.verify))
        if dump and args.subcompactions <= 1:           # the single job is the e2e result
            dump_counters(dumps, "e2e", res[-1][0])
            dump_file_sample(dumps, "e2e_data", out_data[:int(res[-1][0]["output_data_file_size"])])
            dump_file_sample(dumps, "e2e_meta", out_meta[:int(res[-1][0]["output_meta_file_size"])])
        if args.subcompactions > 1:
            files = [(s.meta_view(), s.data_view()) for s in ssts]

            def step_sub():
                r = pkg.compact_files(files, max_subcompactions=args.subcompactions, max_in_flight=args.in_flight,
                                      data_arena=out_data, meta_arena=out_meta, device=local_rank,
                                      verify_checksums=bool(args.verify), **job_kw)
                last_sub[0] = r
                return r.total.as_dict(), sum(o_.data_len + o_.meta_len for o_ in r.outputs), len(r.outputs)

            last_sub = [None]
            sub_s, sres = timed(step_sub, info_steps)
            try:
                sub_check = verify_outputs([(out_meta[o_.meta_offset:o_.meta_offset + o_.meta_len], out_data[o_.data_offset:o_.data_offset + o_.data_len])
                                            for o_ in last_sub[0].outputs if o_.data_len])
            except Exception as ex:
                sub_check = {"error": "%s: %s" % (type(ex).__name__, ex)}
            assert sres[-1][0]["num_input_records"] == n_entries, "subcompactions must see every input entry once"
            range_files = {"value": round(in_bytes * world * info_steps / sub_s / 1e9, 4), "unit": "GB/s", "steps": info_steps,
                           "ms_per_step": round(sub_s / info_steps * 1e3, 2), "output_files": int(sres[-1][2]),
                           "output_file_bytes": int(sres[-1][1]), "output_check": sub_check,
                           "gpu_ms_per_step": round(sres[-1][0]["gpu_seconds"] * 1e3, 2),
                           "mode": "ybgpu_compact_files, one output SST per key range (the shape CompactionJob gives "
                                   "subcompactions, compaction_job.cc:1128-1131) — NOT the headline: DocDB writes one file"}

            # HEADLINE: ONE output table, the shape DocDB's single-level universal compaction (and the reference arm)
            # writes. ybgpu_compact_files_one_table: the key ranges run pipelined, every range's data blocks go
            # device->host straight to their final position in the one data file, and the one metadata file
            # (rebased multi-level index, all filter blocks + one filter index, summed properties) is assembled in key
            # order while later ranges still run — all inside the timed region.
            one_meta = np.empty(2 * out_meta.size + (1 << 20), np.uint8)
            one_meta[::4096] = 0                        # touch the pages once, outside the timed region

            def step_one_table():
                data, meta, res_, tot = pkg.compact_files_one_table(files, max_subcompactions=args.subcompactions, max_in_flight=args.in_flight,
                                                                    data_out=out_data, meta_out=one_meta, device=local_rank,
                                                                    verify_checksums=bool(args.verify), **job_kw)
                return tot.as_dict(), int(data.size), int(meta.size), int(res_.num_pieces), meta
            ot_s, ores = timed(step_one_table, args.steps)
            st_d, data_bytes, meta_bytes, n_pieces, meta = ores[-1]
            off, sz, _ = pkg.sst_block_handles(meta)     # the product's own reader walks the merged index
            assert len(off) == st_d["num_output_data_blocks"] and int(off[-1] + sz[-1]) + 5 == data_bytes
            assert st_d["num_input_records"] == n_entries
            one_check = verify_outputs([(meta, out_data[:data_bytes])])
            if dump:
                dump_counters(dumps, "e2e", st_d)
                dump_file_sample(dumps, "e2e_data", out_data[:data_bytes])
                dump_file_sample(dumps, "e2e_meta", meta)
            e2e = {"value": round(in_bytes * world * args.steps / ot_s / 1e9, 4), "unit": "GB/s", "steps": args.steps,
                   "h2d_bytes_per_step": int(st_d["h2d_bytes"]), "d2h_bytes_per_step": int(st_d["d2h_bytes"]),
                   "ms_per_step": round(ot_s / args.steps * 1e3, 2), "pinned_inputs": all(ok for _, ok in pinned),
                   "output_files": 1, "output_file_bytes": int(data_bytes + meta_bytes), "verify_checksums": bool(args.verify),
                   "mode": "ONE output table: ybgpu_compact_files_one_table (%d key ranges, %d in flight on private streams, data pieces "
                           "copied to their final offsets, metadata file assembled while later ranges run)" % (n_pieces, args.in_flight),
                   "pieces": int(n_pieces), "data_blocks": int(len(off)), "output_check": one_check,
                   "gpu_ms_per_step": round(st_d["gpu_seconds"] * 1e3, 2),
                   "pcie_ceiling_gbs": ceiling,
                   "range_files": range_files,
                   "single_job": single}
            del one_meta
            if isinstance(ceiling, dict) and "both" in ceiling and ceiling["both"]:
                # the step moves in_bytes in and about as much out at once; "both" is the per-direction rate of exactly that
                e2e["frac_of_pcie_ceiling"] = round(e2e["value"] / ceiling["both"], 3)
        for v, ok in pinned:
            if ok:
                cudart.cudaHostUnregister(v.ctypes.data)
        del out_data, out_meta
    if dump:
        write_dumps(args.dump_outputs, dumps)

    # ---- BASELINE configs[2] and configs[3] as sub-results (the bench line itself is configs[1]) ----
    extra = {}
    if not args.no_extra_configs and args.workload == "config2":
        pinned = None
        del ssts, handles
        torch.cuda.empty_cache()
        try:   # configs[2]: 64 tablets x 4-way x 10 M keys across 8 GPUs = 8 tablets per GPU, one after the other
            tabs = []
            t0 = time.perf_counter()
            for t in range(args.c3_tablets):
                tid = rank * args.c3_tablets + t
                c3 = pkg.GenConfig(seed=1000 + tid, num_rows=args.c3_rows, cols=1, versions=1, num_files=4, value_len=VALUE_LEN,
                                   row_offset=tid * args.c3_rows, hash_rows_total=args.c3_rows * args.c3_tablets * world)
                ts = pkg.generate_ssts(c3, max_threads=4)
                tabs.append((ts, [read_handles(pkg, s_) for s_ in ts]))
            c3_gen = time.perf_counter() - t0
            c3_in = sum(s_.raw_bytes for ts, _ in tabs for s_ in ts)
            c3_entries = sum(s_.num_entries for ts, _ in tabs for s_ in ts)
            def to_dev(v):
                t_ = torch.empty(v.size + 64, dtype=torch.uint8, device="cuda")
                t_[16:16 + v.size].copy_(torch.from_numpy(v))
                return t_
            dev = [[to_dev(s_.data_view()) for s_ in ts] for ts, _ in tabs]

            def c3_step():
                sts = []
                for (ts, hs), dts in zip(tabs, dev):
                    job = pkg.GpuCompactionJob(device=local_rank, verify_checksums=bool(args.verify), cuda_stream=stream_ptr, **job_kw)
                    for t_, s_, (off, sz) in zip(dts, ts, hs):
                        job.add_input_device(t_.data_ptr() + 16, s_.data_view().size, off, sz)
                    sts.append(job.run().as_dict())
                    job.close()
                return sts
            c3_step()
            c3_steps = min(args.steps, 3)
            barrier()
            t0 = time.perf_counter()
            c3_stats = [c3_step() for _ in range(c3_steps)]
            barrier()
            dt = time.perf_counter() - t0
            te = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            dt = float(te.item())
            flat = [x for st_ in c3_stats for x in st_]
            gpu_s = sum(x["gpu_seconds"] for x in flat) / c3_steps
            c3_out = sum(x["total_output_raw_key_bytes"] + x["total_output_raw_value_bytes"] for x in c3_stats[-1])
            ach = (c3_in + c3_out) / gpu_s / 1e9
            extra["configs[2]"] = {
                "workload": "64 tablets x 4-way compaction, 10M keys each, tablet-sharded across 8 GPUs: %d tablets x %d entries per GPU, %d GPU(s) in this run, "
                            "inputs resident in HBM, jobs back to back on one stream" % (args.c3_tablets, args.c3_rows, world),
                "value": round(c3_in * world * c3_steps / dt / 1e9, 2), "unit": "GB/s", "mkeys_per_s": round(c3_entries * world * c3_steps / dt / 1e6, 1),
                "ms_per_step": round(dt / c3_steps * 1e3, 2), "steps": c3_steps, "tablets_per_gpu": args.c3_tablets,
                "entries_per_gpu": int(c3_entries), "verify_checksums": bool(args.verify), "generate_s": round(c3_gen, 1),
                "roofline": {"bound": "hbm", "scope": "whole pipeline", "algorithmic_bytes": int(c3_in + c3_out), "gpu_ms": round(gpu_s * 1e3, 2),
                             "achieved": round(ach, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(ach / hbm_peak, 4)}}
            del tabs, dev
            torch.cuda.empty_cache()
        except Exception as ex:
            extra["configs[2]"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        if world == 1:
            try:   # configs[3]: MVCC-heavy, 20 versions per key, the history cutoff drops 18 of 20 (90 %)
                live = args.c4_rows // 20
                c4 = pkg.GenConfig(seed=77, num_rows=live, cols=1, versions=20, num_files=NUM_FILES, value_len=VALUE_LEN)
                t0 = time.perf_counter()
                s4 = pkg.generate_ssts(c4, max_threads=NUM_FILES)
                c4_gen = time.perf_counter() - t0
                h4 = [read_handles(pkg, s_) for s_ in s4]
                kw4 = dict(job_kw, cutoff_ht=((c4.base_micros + 18 * 1000 + 500) << 12))
                c4_in = sum(s_.raw_bytes for s_ in s4)
                c4_entries = sum(s_.num_entries for s_ in s4)
                c4_steps = min(args.steps, 3)
                c4_s, c4_stats, _, _ = resident_arm(pkg, torch, s4, h4, local_rank, stream_ptr, kw4, args.verify, c4_steps, 1, barrier, world, dist)
                roof = pipeline_roofline(c4_stats, c4_in, hbm_peak, c4_steps)
                extra["configs[3]"] = {
                    "workload": "MVCC-heavy: 20 versions/key, history_cutoff drops 90%%, %d live keys (%d entries, %.1f GB raw) resident on 1 GPU; "
                                "BASELINE names 50M live keys = 1 G entries = 310 GB, which exceeds the 180 GB of HBM" % (live, c4_entries, c4_in / 1e9),
                    "value": round(c4_in * c4_steps / c4_s / 1e9, 2), "unit": "GB/s", "mkeys_per_s": round(c4_entries * c4_steps / c4_s / 1e6, 1),
                    "ms_per_step": round(c4_s / c4_steps * 1e3, 2), "steps": c4_steps, "entries": int(c4_entries),
                    "output_entries": int(c4_stats[-1]["num_output_records"]), "dropped_fraction": round(1.0 - c4_stats[-1]["num_output_records"] / c4_entries, 4),
                    "verify_checksums": bool(args.verify), "generate_s": round(c4_gen, 1),
                    "roofline": dict(roof, bound="hbm", scope="whole pipeline")}
                del s4, h4
                torch.cuda.empty_cache()
            except Exception as ex:
                extra["configs[3]"] = {"error": "%s: %s" % (type(ex).__name__, ex)}

    run_c5 = world > 1 and not args.no_extra_configs and args.workload == "config2"

    def finish(line):
        """Rank 0 prints the one JSON line — after the key-range sharded sub-result (configs[4], N > 1 only), which all
        ranks run under a watchdog: a rank that fails or hangs inside the exchange must not cost the whole line."""
        printed = threading.Event()

        def emit_once(c5=None):
            if rank == 0 and not printed.is_set():
                printed.set()
                if c5 is not None:
                    line.setdefault("configs", {})["configs[4]"] = c5
                emit_json_line(line)
        if run_c5:
            def bail():
                emit_once({"error": "no result within %.0f s (watchdog)" % args.c5_timeout})
                os._exit(0)
            timer = threading.Timer(args.c5_timeout, bail)
            timer.daemon = True
            timer.start()
            failed = False
            try:
                c5 = config5_sharded(args, pkg, torch, dist, rank, world, local_rank, job_kw, hbm_peak, barrier)
            except Exception as ex:
                c5, failed = {"error": "%s: %s" % (type(ex).__name__, ex)}, True
            timer.cancel()
            emit_once(c5)
            if failed:
                os._exit(0)                     # the other ranks may be stuck in a collective: do not wait for them
        else:
            emit_once()
        if world > 1:
            dist.destroy_process_group()

    if rank != 0:
        finish(None)
        return

    # dominant kernel = longest phase; its algorithmic bytes (DESIGN.md "Roofline accounting")
    names = pkg.PHASE_NAMES
    # The dominant KERNEL: ingest (verify + decode) and merge phases are one kernel each; the encode phase is ~25
    # launches of which the block assembler is timed separately.
    kernel_s = {"ingest(verify+decode)": phases[0] + phases[1], "k_merge_filter": phases[3], "k_encode": enc_kernel_s}
    kernel_alg = {"ingest(verify+decode)": float(in_bytes),         # must read every input byte once
                  "k_merge_filter": float(in_bytes + out_bytes),    # charged the whole path (it moves only keys)
                  "k_encode": out_bytes * 2.0}                      # read each survivor once, write it once
    dom_kernel = max(kernel_s, key=lambda k: kernel_s[k])
    dom_bytes = kernel_alg[dom_kernel]
    achieved = dom_bytes / kernel_s[dom_kernel] / 1e9 if kernel_s[dom_kernel] > 0 else 0.0
    # DRAM traffic of that kernel: NOT measured in this run — read from the committed `ncu --set full` capture of this
    # same command (profiles/), labelled so
    traffic, traffic_src = None, None
    try:
        if args.workload == "config2" and args.rows == DEFAULT_ROWS:
            for fn in ("r02_ncu_full_100m.json", "r01_ncu_full_100m.json"):
                path = os.path.join(ROOT, "profiles", fn)
                if not os.path.exists(path):
                    continue
                prof = json.load(open(path))["kernels"]
                want = {"ingest(verify+decode)": ("k_ingest", "k_decode"), "k_merge_filter": ("k_merge_filter",), "k_encode": ("k_encode",)}[dom_kernel]
                for name, kd in prof.items():
                    if name.startswith(want):
                        def gb(x):
                            v = float(x["value"]); return v * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[x["unit"]]
                        traffic = int(gb(kd["dram__bytes_read.sum"]) + gb(kd["dram__bytes_write.sum"]))
                        traffic_src = "profiles/%s (%s), committed capture, not measured in this run" % (fn, name)
                        break
                if traffic is not None:
                    break
    except Exception:
        traffic = None
    value = in_bytes * world * args.steps / total_s / 1e9
    line = {
        "metric": "compaction GB/s (input bytes merged)", "value": round(value, 3), "unit": "GB/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(total_s / args.steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": (WORKLOAD if args.rows == DEFAULT_ROWS else WORKLOAD + " (scaled to %d entries)" % args.rows)
                   if args.workload == "config2" else
                   "MVCC-heavy: 20 versions/key, history_cutoff drops 90%%, %d live keys, 1 GPU (8 input files)" % nrows,
                   "output_entries_per_gpu": int(stats[-1]["num_output_records"]),
                   "entries_per_gpu": int(n_entries), "input_raw_bytes_per_gpu": int(in_bytes),
                   "input_file_bytes_per_gpu": int(file_bytes), "tablets": world,
                   "parallelism": "tablet-per-GPU, no collective",
                   "verify_checksums": bool(args.verify),
                   "host_placement": {"numa_node": numa_node, "cpus": numa_cpus},
                   "output": "split SST: data blocks + CRC32C, multi-level index, DocKeyV3 bloom filter blocks (64 KB), properties, footer",
                   "l2": "inputs (%.1f GB) far larger than the 126 MB L2" % (file_bytes / 1e9)},
        "mkeys_per_s": round(n_entries * world * args.steps / total_s / 1e6, 2),
        "gpu_launches": int(launches),
        "clocks": clock_info,
        "value_no_verify": {"value": round(in_bytes * world * nv_steps / nv_s / 1e9, 3), "unit": "GB/s", "steps": nv_steps,
                            "ms_per_step": round(nv_s / nv_steps * 1e3, 3),
                            "note": "input block checksums NOT verified (work the reference does is skipped): informational only"},
        "roofline": {"bound": "hbm", "kernel": dom_kernel, "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
                     "frac": round(achieved / hbm_peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_kind,
                     "kernel_ms": round(kernel_s[dom_kernel] * 1e3, 3), "algorithmic_bytes_per_launch": int(dom_bytes),
                     "kernels_ms": {k: round(v * 1e3, 3) for k, v in kernel_s.items()},
                     "pipeline": pipeline_roofline(stats, in_bytes, hbm_peak, args.steps),
                     "phase_ms": {names[i]: round(phases[i] * 1e3, 3) for i in range(5)}},
        "setup": {"generate_s": round(gen_s, 1)},
        "host_ms_per_step": host_ms,
    }
    if e2e:
        line["e2e"] = e2e
    if dump:
        line["dump_outputs"] = dump_info
    if extra:
        line["configs"] = extra
    if not args.no_cpu_baseline:
        base, parity = cpu_baseline(args, pkg, local_rank)
        line["cpu_baseline"] = base
        line["parity_check"] = parity
    finish(line)


def config5_sharded(args, pkg, torch, dist, rank, world, local_rank, job_kw, hbm_peak, barrier):
    """BASELINE configs[4]: ONE oversized tablet, 32 input files, key-range sharded across the GPUs through
    ybgpu_compact_range_sharded (C++ over NCCL: splitters all-gathered, block slices exchanged with chunked grouped
    ncclSend / ncclRecv over NVLink, every rank compacting its key range). All ranks call this; returns the
    sub-result on rank 0. Scaled: --c5-rows-per-gpu entries per GPU (the 1 TB of BASELINE does not fit 8 x 180 GB
    together with the outputs; the `rounds` mechanism that bounds HBM use is exercised by the tests)."""
    n_files = 32
    total_rows = args.c5_rows_per_gpu * world
    cfg = pkg.GenConfig(seed=5, num_rows=total_rows, cols=1, versions=1, num_files=n_files, value_len=VALUE_LEN)
    mine = [f for f in range(n_files) if f % world == rank]
    t0 = time.perf_counter()
    ssts = pkg.generate_sst_files(cfg, mine, max_threads=len(mine))
    gen_s = time.perf_counter() - t0
    files = [(s_.meta_view(), s_.data_view()) for s_ in ssts]
    local_in = sum(s_.raw_bytes for s_ in ssts)
    local_entries = sum(s_.num_entries for s_ in ssts)
    local_file_bytes = sum(int(d.size) for _, d in files)
    cudart = torch.cuda.cudart()
    pinned = [int(cudart.cudaHostRegister(d.ctypes.data, d.size, 0)) == 0 for _, d in files]
    tot = torch.tensor([float(local_in), float(local_entries), float(local_file_bytes)], dtype=torch.float64, device="cuda")
    dist.all_reduce(tot)
    total_in, total_entries, total_file_bytes = (float(x) for x in tot.tolist())
    out_cap = int(total_file_bytes / world * 1.5) + (256 << 20)
    out_data = torch.empty(out_cap, dtype=torch.uint8, pin_memory=True).numpy()
    out_meta = torch.empty(max(64 << 20, out_cap // 50), dtype=torch.uint8, pin_memory=True).numpy()
    uid = [pkg.range_comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    comm = pkg.RangeComm(uid[0], rank, world, local_rank)
    results = []
    steps = min(args.steps, 2)
    dts = []
    for it in range(1 + steps):                      # one warm-up (communicator set-up, allocator) + `steps` timed
        barrier()
        t0 = time.perf_counter()
        data, meta, res, st = comm.compact(files, rounds=1, chunk_bytes=64 << 20, data_out=out_data, meta_out=out_meta,
                                           verify_checksums=bool(args.verify), **job_kw)
        torch.cuda.synchronize()
        barrier()
        dt = time.perf_counter() - t0
        te = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        if it:
            dts.append(float(te.item()))
            results.append((res, st))
    res, st = results[-1]
    mine_stats = torch.tensor([float(st.num_input_records), float(st.num_output_records), float(res.sent_to_peers_bytes),
                               float(res.exchange_seconds), float(st.gpu_seconds), float(res.data_len)], dtype=torch.float64, device="cuda")
    summed = mine_stats.clone()
    dist.all_reduce(summed)
    mx = mine_stats.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    comm.close()
    for (_, d), ok in zip(files, pinned):
        if ok:
            cudart.cudaHostUnregister(d.ctypes.data)
    if rank != 0:
        return None
    dt = sum(dts) / len(dts)
    s_in, s_out, nvl, _, _, s_dlen = (float(x) for x in summed.tolist())
    _, _, _, ex_max, gpu_max, _ = (float(x) for x in mx.tolist())
    assert int(s_in) == int(total_entries), "the ranks' key ranges must cover every input entry exactly once"
    return {
        "workload": "single tablet, 32-way major compaction, key-range-sharded across %d GPUs with one NCCL exchange: %d entries "
                    "(%.1f GB raw, %.1f GB of files) in total, %d per GPU; host files in, one host table per rank out" % (
                        world, int(total_entries), total_in / 1e9, total_file_bytes / 1e9, args.c5_rows_per_gpu),
        "value": round(total_in / dt / 1e9, 2), "unit": "GB/s", "mkeys_per_s": round(total_entries / dt / 1e6, 1),
        "ms_per_step": round(dt * 1e3, 1), "steps": steps, "timing": "host wall clock between barriers, max over ranks (includes "
        "host->device staging of the inputs and device->host copy of the outputs)",
        "exchange": {"nvlink_bytes": int(nvl), "seconds_max_rank": round(ex_max, 4),
                     "aggregate_gbs": round(nvl / ex_max / 1e9, 1) if ex_max > 0 else None,
                     "mechanism": "ncclSend/ncclRecv grouped per 64 MB chunk, counts all-gathered first, staged from pinned host memory"},
        "gpu_seconds_max_rank": round(gpu_max, 4), "output_entries": int(s_out), "output_data_bytes": int(s_dlen),
        "ranges": int(res.num_ranges), "verify_checksums": bool(args.verify), "generate_s": round(gen_s, 1)}


def read_handles(pkg, sst):
    """Data-block handles of a generated SST, via the product's host meta reader."""
    off, sz, _ = pkg.sst_block_handles(sst.meta_view())
    return off, sz


if __name__ == "__main__":
    main()
