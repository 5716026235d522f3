#!/usr/bin/env python3
"""Headline benchmark: Gbases/s of the TREW scan-and-count hot path (`trew short 5 32`) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* is one pass of the hot path over one file-sized set of synthetic reads of BASELINE.json's configs[1] shape
(200 M x 150 bp, ~1 % TTAGGG reads, MIN_MER 5, MAX_MER 32), sharded over the N GPUs (strong scaling: 200 M / N per
GPU, SURVEY 8(d); --scaling weak puts 200 M on every GPU): reset the count table, scan every resident batch (screen,
decide, the two exact kernels per batch), compact the table, copy it to the host and -- for N > 1 -- merge the
per-rank tables exactly over NCCL.

  value      whole-job Gbases/s with the packed reads already resident in HBM (generated on the device), timed with
             CUDA events on the scan stream, max over ranks.  Batches of 16 M reads: 12 GB of input per pass at N = 1,
             far larger than L2, so no flush is needed between iterations.
  e2e        the same metric through the reference-facing C ABI with HOST buffers, all N GPUs driven by one process:
             4-line FASTQ chunks + sequence-line offsets (the reference's QueueData) -> trew_multi_submit_chunk (host
             packing on every core, pinned staging, cudaMemcpyAsync, kernels, chunks dealt round-robin over the GPUs)
             -> trew_multi_finish (peer copies + union on the first GPU, tables back on the host), wall clock.
  e2e_file   from FASTQ files on disk (plain / .gz / BGZF) through trew_multi_process_file, and the `trew` binary itself.
  roofline   the scan pipeline of one batch (screen + decide + exact kernels): algorithmic bytes of the batch / the
             CUDA-event time of its kernels, against the measured HBM copy bandwidth in MEASURED_PEAKS.json; per-kernel
             figures and the committed ncu pipe utilisation beside it (the path is instruction-bound, not HBM-bound).
  configs    the other BASELINE.json shapes (paired, long, 3..64) on the same GPU, one batch each (N = 1 only).
  cpu_baseline  the reference's own CPU path (oracle/_ref, compiled from the unmodified sources) on the
             box's host cores, on a bounded sample of the same workload.  Reported, not the target.

--impl reference times only that CPU path (rank 0; other ranks exit) and prints the same JSON shape.

--dump-outputs DIR writes the tables the last timed step returned (rank 0) as float64 .npy files, so that two builds
can be compared output for output: the inputs are seeded, identical from run to run for the same arguments.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "Gbases/s for trew short 5 32 at 1/2/4/8 B200; % of HBM roofline"
READ_LEN = 150
BATCH_READS = 25_000_000   # 3.75 G bases per resident batch (bit offsets are 32-bit: < 4.29 G); larger batches amortise the exact kernels' tails
BYTES_PER_READ = 4 + 3 * READ_LEN / 8.0  # offsets + three bit-planes (DESIGN.md, "algorithmic bytes")
SYNTH = dict(tel_ppm=10000, half_ppm=2000, n_ppm=1000, sub_ppm=10000)


def workload_name(total_reads, world=1, strong=True):
    how = "in total" if strong else "(%d M per GPU, weak scaling)" % (total_reads // max(1, world) // 1_000_000)
    return ("synthetic short-read single-end: %d M x %d bp reads %s with ~1%% TTAGGG-repeat reads, "
            "MIN_MER=5 MAX_MER=32" % (total_reads // 1_000_000, READ_LEN, how))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe): one nvidia-smi
    process streaming a sample every 50 ms between start() and stop()."""

    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.samples = []
        self.window = (0.0, float("inf"))   # wall-clock bounds of the timed region

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return
        try:
            self.proc.terminate()
            out = self.proc.communicate(timeout=5)[0].decode()
        except Exception:
            out = ""
        import datetime
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                ts = None
            if ts is None or self.window[0] - 0.05 <= ts <= self.window[1] + 0.05:
                self.samples.append(f[1:])

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        power = sorted(float(s[2]) for s in self.samples if s[2].replace(".", "", 1).isdigit())
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm), "power_w_max": power[-1] if power else None}


def load_issue_profile():
    """Per-kernel pipe utilisation from the committed ncu run (profiles/issue_profile.json, written by
    tools/ncu_summary.py from an `ncu --set full` capture of tools/profile_scan.py): the evidence for `limiter`."""
    p = os.path.join(ROOT, "profiles", "issue_profile.json")
    try:
        return json.load(open(p))
    except Exception:
        return None


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------
# the reference's CPU path (oracle/_ref): only for cpu_baseline / --impl reference
# ---------------------------------------------------------------------------------------------

def write_sample_fastq(path, n_reads, seed=1):
    from trew_b200 import synth
    with open(path, "wb") as f:
        done = 0
        while done < n_reads:
            m = min(250_000, n_reads - done)
            mat = synth.config_short(seed + done, m, READ_LEN, telomeric=SYNTH["tel_ppm"] / 1e6,
                                     half_telomeric=SYNTH["half_ppm"] / 1e6, n_rate=SYNTH["n_ppm"] / 1e6,
                                     sub=SYNTH["sub_ppm"] / 1e6)
            f.write(synth.fastq_matrix_bytes(mat))
            done += m


def time_reference(sample_fastq, cores):
    from oracle.oracle import REF_BIN
    t0 = time.perf_counter()
    subprocess.run([REF_BIN, "short", "5", "32", sample_fastq, "-t", str(cores), "-q", "1024"], check=True,
                   stdout=subprocess.DEVNULL)
    return time.perf_counter() - t0


def reference_available():
    from oracle.oracle import REF_BIN
    return os.path.exists(REF_BIN)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    cores = os.cpu_count() or 1
    line = {"metric": METRIC, "unit": "Gbases/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "impl": "reference", "config": {"workload": workload_name(args.reads if args.scaling == "strong" else args.reads * args.gpus,
                                                                     args.gpus, args.scaling == "strong")}}
    if not reference_available():
        line["unavailable"] = "oracle/_ref/trew_ref missing (reference not compiled into this tree)"
        return line
    tmp = tempfile.mkdtemp(prefix="trew_ref_")
    try:
        # calibrate on 100k reads, then size the sample so warmup + steps stay within ~150 s
        cal = os.path.join(tmp, "cal.fastq")
        write_sample_fastq(cal, 100_000)
        t_cal = max(time_reference(cal, cores) - 0.6, 0.05)  # ~0.6 s of table setup at -m 12
        budget = 150.0 / max(1, args.steps + args.warmup)
        n = int(min(2_000_000, max(100_000, 100_000 * budget / t_cal)))
        sample = os.path.join(tmp, "sample.fastq")
        write_sample_fastq(sample, n)
        for _ in range(args.warmup):
            time_reference(sample, cores)
        times = [time_reference(sample, cores) for _ in range(args.steps)]
        total = sum(times)
        value = n * READ_LEN * len(times) / total / 1e9
        sample_desc = ("%d reads of the same distribution (numpy generator) as plain FASTQ, "
                       "`trew_ref short 5 32 -t %d -q 1024`, wall clock" % (n, cores))
        line.update({"value": value, "ms_per_step": 1e3 * total / len(times),
                     "cpu_baseline": {"value": value, "unit": "Gbases/s", "cores": cores, "kind": "reference", "sample": sample_desc},
                     "e2e": {"value": value, "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "gpu_launches": 0})
        return line
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------

DUMP_MAX_ROWS = 1_000_000   # 7 float64 columns: 56 MB at most


def _mix64(x):
    """splitmix64's finaliser on a uint64 array (wrapping arithmetic)."""
    x = x ^ (x >> np.uint64(30))
    x = x * np.uint64(0xbf58476d1ce4e5b9)
    x = x ^ (x >> np.uint64(27))
    x = x * np.uint64(0x94d049bb133111eb)
    return x ^ (x >> np.uint64(31))


def dump_outputs(rows, out_dir):
    """The entries of a step (sorted by (table, k, seq)) as DIR/{table,k,seq,count}.npy in float64, every value exact:
    seq is split into its four 32-bit words, least significant first (n x 4).  Above DUMP_MAX_ROWS entries the sample
    is the DUMP_MAX_ROWS keys with the smallest seeded hash of (table, k, seq), still in table order: it depends on the
    keys alone, so two builds whose tables differ in a few keys write samples that differ in about as few rows.
    Returns what was written."""
    n = int(rows.shape[0])
    idx = np.arange(n)
    if n > DUMP_MAX_ROWS:
        meta = (rows["table"].astype(np.uint64) << np.uint64(8)) | rows["k"].astype(np.uint64)
        with np.errstate(over="ignore"):
            h = _mix64(_mix64(_mix64(meta ^ np.uint64(0x9e3779b97f4a7c15)) ^ rows["seq_lo"]) ^ rows["seq_hi"])
        idx = np.sort(np.argpartition(h, DUMP_MAX_ROWS)[:DUMP_MAX_ROWS])
    r = rows[idx]
    mask = np.uint64(0xffffffff)
    seq = np.stack([r["seq_lo"] & mask, r["seq_lo"] >> np.uint64(32), r["seq_hi"] & mask, r["seq_hi"] >> np.uint64(32)], axis=1)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"table": r["table"], "k": r["k"], "seq": seq, "count": r["count"]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))
    return {"dir": os.path.abspath(out_dir), "rows": n, "rows_written": int(idx.shape[0]),
            "arrays": {name: list(a.shape) for name, a in arrays.items()}}


def fastq_chunk(api, synth, seed, n_reads):
    """One raw chunk exactly as the reference's read_fastq_thread pushes it (QueueData, src/kmer.h:93-96): 4-line
    FASTQ text (header, sequence, '+', quality) plus the inclusive (st, nd) offsets of the sequence lines."""
    mat = synth.config_short(seed, n_reads, READ_LEN, telomeric=SYNTH["tel_ppm"] / 1e6, half_telomeric=SYNTH["half_ppm"] / 1e6,
                             n_rate=SYNTH["n_ppm"] / 1e6, sub=SYNTH["sub_ppm"] / 1e6)
    buf = np.frombuffer(synth.fastq_matrix_bytes(mat), dtype=np.uint8)
    rec = 3 + READ_LEN + 1 + 2 + READ_LEN + 1          # '@r\n' + seq + '\n' + '+\n' + qual + '\n'
    st = np.arange(n_reads, dtype=np.int64) * rec + 3
    locs = np.empty((n_reads, 2), dtype=np.int32)
    locs[:, 0] = st
    locs[:, 1] = st + READ_LEN - 1
    return buf, locs


def run_ours(args):
    import torch
    import torch.distributed as dist
    from trew_b200 import api, merge, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    host_pg = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints one JSON line
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        host_pg = dist.new_group(backend="gloo")   # host-side waits that keep the other ranks' GPUs idle
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    strong = args.scaling == "strong"
    ctx = api.DeviceContext(api.MODE_SHORT, 5, 32, device=local_rank, n_staging=2, staging_bytes=16 << 20, host_threads=2)

    # ---- device-resident workload.  strong: configs[1]'s 200 M reads are sharded over the ranks (SURVEY 8(d): shard =
    # 200 M / G); weak: every rank holds args.reads reads. -------------------------------------------------------------
    reads_rank = args.reads // world if strong else args.reads
    handles, reads_left, i = [], reads_rank, 0
    while reads_left > 0:
        n = min(BATCH_READS, reads_left)
        handles.append((ctx.synth_resident(1 + 1000 * rank + i, n, READ_LEN, **SYNTH), n))
        reads_left -= n
        i += 1
    total_reads = reads_rank * world

    # a step ends with the tables of the "file" on the host: the rows that can reach the report of a one-file run (groups
    # with a class total >= 10, trew_dev_set_report_filter) -- what `trew short 5 32 FILE` copies; the same step with every
    # row (the six raw maps) is timed beside it as full_tables_ms_per_step
    ctx.set_report_filter(0 if args.full_tables else 10)

    def step():
        ctx.reset()
        for h, _ in handles:
            ctx.scan_resident(h)
        # sync + compaction kernel + D2H of the tables (+ exact NCCL merge across ranks for N > 1)
        return merge.finish_merged(ctx, device) if world > 1 else ctx.finish_view()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()   # nvidia-smi needs a moment to come up: started before the warm-up, filtered to the timed region
    for _ in range(args.warmup):
        step()
    ctx.kernel_times()  # drop warm-up kernel times
    launches0 = ctx.stats().kernel_launches
    barrier()
    ctx.timer_start()
    t0 = time.perf_counter()
    wall0 = time.time()
    for _ in range(args.steps):
        rows = step()
    dev_ms = ctx.timer_stop()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    if rank == 0:
        sampler.window = (wall0, time.time())
        sampler.stop()
        table_rows = int(rows.shape[0])
        # rows is a view of the library's entries: written out before the next step replaces them
        dumped = dump_outputs(rows, args.dump_outputs) if args.dump_outputs else None
    # finish() and the merge run on the host between the event pair, so the event time covers the step
    ms = max_over_ranks(max(dev_ms, 0.0))
    wall_ms = max_over_ranks(wall_ms)
    screen_ms, decide_ms, exact_ms, n_scans = ctx.kernel_times()
    st = ctx.stats()
    launches = st.kernel_launches - launches0
    # the same step returning every row of the six maps
    ctx.set_report_filter(0)
    step()
    barrier()
    ctx.timer_start()
    for _ in range(3):
        full_rows = step()
    full_ms = max_over_ranks(ctx.timer_stop()) / 3
    barrier()
    ctx.kernel_times()
    full_table_rows = int(full_rows.shape[0]) if rank == 0 else 0
    value = total_reads * READ_LEN * args.steps / (ms * 1e-3) / 1e9
    survivor_fraction = st.survivors / max(1, st.units)

    # ---- end to end through the C ABI with HOST buffers, all GPUs of the box driven by ONE process (trew_multi: one
    # context per device, one packing pool on every core, chunks dealt round-robin, merge on the first device).  Under
    # torchrun rank 0 runs it; the other ranks wait on the host. -------------------------------------------------------
    e2e = None
    extra = {}
    if rank == 0:
        devices = list(range(world))
        multi = api.MultiContext(api.MODE_SHORT, 5, 32, devices=devices, n_staging=3, staging_bytes=96 << 20)
        chunk_reads = min(args.e2e_reads, 1_000_000)
        buf, locs = fastq_chunk(api, synth, 7, chunk_reads)
        reps = max(world, args.e2e_reads * world // chunk_reads)     # chunks per step: args.e2e_reads per GPU
        e2e_reads = reps * chunk_reads

        def e2e_step():
            multi.reset()
            for _ in range(reps):
                multi.submit_chunk(buf, locs)
            return multi.finish_view()

        for _ in range(max(1, min(args.warmup, 2))):
            e2e_step()
        st1 = multi.stats()
        t0 = time.perf_counter()
        e2e_steps = max(1, min(args.steps, 5))
        for _ in range(e2e_steps):
            e2e_step()
        e2e_s = time.perf_counter() - t0
        st2 = multi.stats()
        pack_ms = st2.host_pack_ms - st1.host_pack_ms
        e2e = {"value": e2e_reads * READ_LEN * e2e_steps / e2e_s / 1e9, "unit": "Gbases/s",
               "h2d_bytes_per_step": int((st2.h2d_bytes - st1.h2d_bytes) / e2e_steps),
               "d2h_bytes_per_step": int((st2.d2h_bytes - st1.d2h_bytes) / e2e_steps),
               "reads_per_step": int(e2e_reads), "steps": e2e_steps, "gpus": world,
               "path": "4-line FASTQ chunk + sequence-line offsets (QueueData) -> trew_multi_submit_chunk -> trew_multi_finish, one process",
               "host_pack": {"seconds_per_step": pack_ms * 1e-3 / e2e_steps,
                             "share_of_step": pack_ms * 1e-3 / e2e_s,
                             "ascii_gbytes_per_s": (st2.host_pack_bytes - st1.host_pack_bytes) / max(pack_ms * 1e-3, 1e-9) / 1e9,
                             "threads": os.cpu_count(),
                             "note": "the submitting thread packs one chunk at a time with every core; the GPUs only see the packed "
                                     "planes, so this share is the host bound of the end-to-end path"}}
        if not args.no_cpu_baseline:
            extra["e2e_file"] = file_e2e(multi, api, synth, world)
        multi.close()
    if host_pg is not None:
        dist.barrier(group=host_pg)

    line = None
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        launches_per_scan = len(handles)
        reads_per_launch = reads_rank / len(handles)
        scan_ms = screen_ms + decide_ms + exact_ms
        per_kernel = {}
        for kname, kms in (("trew_screen_kernel", screen_ms), ("trew_filter_kernel", decide_ms),
                           ("trew_exact_thread_kernel + trew_exact_kernel", exact_ms)):
            avg = kms / max(1, n_scans)
            per_kernel[kname] = {"launch_ms": avg, "share_of_scan": kms / scan_ms if scan_ms > 0 else 0.0,
                                 "gbs_alone": BYTES_PER_READ * reads_per_launch / (avg * 1e-3) / 1e9 if avg > 0 else 0.0}
        dominant = max(per_kernel, key=lambda k: per_kernel[k]["launch_ms"])
        # the kernels of a batch are one pipeline over the same packed reads: the bytes a batch streams, over the time
        # all of them take for it
        scan_avg_ms = scan_ms / max(1, n_scans)
        achieved = BYTES_PER_READ * reads_per_launch / (scan_avg_ms * 1e-3) / 1e9 if scan_avg_ms > 0 else 0.0
        line = {
            "metric": METRIC, "value": value, "unit": "Gbases/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_name(total_reads, world, strong), "min_mer": 5, "max_mer": 32, "low": 0.5, "high": 0.8,
                       "reads_per_gpu": reads_rank, "batches_per_gpu_per_step": launches_per_scan, "reads_per_batch": BATCH_READS,
                       "tables": "every row of the six maps" if args.full_tables else "rows of groups with a class total >= 10 (what a one-file report can show)",
                       "l2": "inputs (%.1f GB packed per GPU and pass) exceed L2; no flush" % (BYTES_PER_READ * reads_rank / 1e9),
                       "parallelism": "reads sharded over %d GPU(s), one exact NCCL table merge per step" % world},
            "wall_ms_per_step": wall_ms / args.steps,
            "gpu_launches": int(launches),
            "table_rows": table_rows, "full_table_rows": full_table_rows, "full_tables_ms_per_step": full_ms,
            "kernel_share": {"screen_ms_per_step": screen_ms / args.steps, "decide_ms_per_step": decide_ms / args.steps,
                             "exact_ms_per_step": exact_ms / args.steps, "survivor_fraction": survivor_fraction,
                             "rest_ms_per_step": ms / args.steps - scan_ms / args.steps,
                             "note": "rank 0's kernels; rest = table reset, compaction, sort, D2H and (N > 1) the NCCL merge"},
            "roofline": {"bound": "hbm", "limiter": "instruction issue (XU pipe: POPC), not HBM -- see `issue` and DESIGN.md section 4",
                         "kernel": dominant, "scope": "screen + decide + exact kernels of one batch (one pipeline over the same packed reads)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_read": BYTES_PER_READ,
                         "algorithmic_bytes_per_launch": BYTES_PER_READ * reads_per_launch,
                         "launch_ms": scan_avg_ms,
                         "per_kernel": per_kernel,
                         "issue": load_issue_profile()},
            "e2e": e2e,
            "clocks": sampler.summary(),
        }
        traffic = os.path.join(ROOT, "profiles", "screen_traffic.json")
        if os.path.exists(traffic):
            try:
                t = json.load(open(traffic))   # measured per launch of t["reads_per_launch"] reads; scaled to this run's launches
                line["roofline"]["traffic"] = t["dram_bytes_per_launch"] * reads_per_launch / t["reads_per_launch"]
            except Exception:
                pass
        line.update(extra)
        if dumped is not None:
            line["outputs"] = dumped
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        if world == 1 and not args.no_shapes:
            line["configs"] = other_shapes(api, local_rank, max(1, min(args.steps, 5)), max(1, min(args.warmup, 2)))
    # weak scaling beside it (N > 1): every GPU holds the full 200 M reads
    if world > 1 and strong and not args.no_weak:
        reads_left = args.reads - reads_rank
        while reads_left > 0:
            n = min(BATCH_READS, reads_left)
            handles.append((ctx.synth_resident(1 + 1000 * rank + i, n, READ_LEN, **SYNTH), n))
            reads_left -= n
            i += 1
        ctx.set_report_filter(0 if args.full_tables else 10)
        step()
        barrier()
        ctx.timer_start()
        for _ in range(3):
            step()
        weak_ms = max_over_ranks(ctx.timer_stop()) / 3
        barrier()
        if rank == 0:
            line["weak_scaling"] = {"value": world * args.reads * READ_LEN / (weak_ms * 1e-3) / 1e9, "unit": "Gbases/s",
                                    "ms_per_step": weak_ms, "reads_per_gpu": args.reads,
                                    "note": "the same step with 200 M reads on EVERY GPU (round 1's definition)"}
    for h, _ in handles:
        ctx.free_resident(h)
    merge.forget(ctx)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return line


def other_shapes(api, device_index, steps, warmup):
    """The other BASELINE.json shapes (configs[2..4]) on the same GPU in the same run: one device-generated resident
    batch each, reset -> scan -> table export per step, CUDA events on the scan stream.  Correctness of these shapes
    is the parity tests' business (tests/test_gpu_parity.py checks the same generator against the oracle)."""
    shapes = [
        ("paired_2x150", "synthetic paired-end: 8 M x 2 x 150 bp per batch, both mates of ~1% of the fragments telomeric, "
                         "--paired_end, MIN_MER=5 MAX_MER=32",
         dict(mode=api.MODE_PAIR, mn=5, mx=32, reads=16_000_000, read_len=150, flavor=1, **SYNTH)),
        ("long_15kb", "synthetic long-read: 200 k x 15 kb per batch, 2% with a telomeric 0.5-5 kb end, 0.1% error, "
                      "trew long 5 32 (SLICE 150)",
         dict(mode=api.MODE_LONG, mn=5, mx=32, reads=200_000, read_len=15000, flavor=2, tel_ppm=20000, half_ppm=0,
              n_ppm=100, sub_ppm=1000)),
        ("sweep_3_64", "full period sweep: 8 M x 150 bp per batch as configs[1], MIN_MER=3 MAX_MER=64 (128-bit units)",
         dict(mode=api.MODE_SHORT, mn=3, mx=64, reads=8_000_000, read_len=150, flavor=0, **SYNTH)),
    ]
    out = {}
    for name, desc, kw in shapes:
        ctx = api.DeviceContext(kw["mode"], kw["mn"], kw["mx"], device=device_index)
        try:
            h = ctx.synth_resident(11, kw["reads"], kw["read_len"], tel_ppm=kw["tel_ppm"], half_ppm=kw["half_ppm"],
                                   n_ppm=kw["n_ppm"], sub_ppm=kw["sub_ppm"], flavor=kw["flavor"])

            def one():
                ctx.reset()
                ctx.scan_resident(h)
                return ctx.finish_view()

            for _ in range(max(1, warmup)):
                rows = one()
            ctx.kernel_times()
            ctx.timer_start()
            for _ in range(steps):
                rows = one()
            ms = ctx.timer_stop()
            s_ms, d_ms, e_ms, n = ctx.kernel_times()
            st = ctx.stats()
            bases = kw["reads"] * kw["read_len"]
            bytes_per_batch = 4 * kw["reads"] + 3 * bases / 8.0
            scan_ms = (s_ms + d_ms + e_ms) / max(1, n)
            out[name] = {"workload": desc, "value": bases * steps / (ms * 1e-3) / 1e9, "unit": "Gbases/s", "ms_per_step": ms / steps,
                         "kernel_share": {"screen_ms": s_ms / max(1, n), "decide_ms": d_ms / max(1, n), "exact_ms": e_ms / max(1, n),
                                          "survivor_fraction": st.survivors / max(1, st.units)},
                         "scan_gbs": bytes_per_batch / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0,
                         "table_rows": int(rows.shape[0])}
            ctx.free_resident(h)
        finally:
            ctx.close()
    return out


def file_e2e(multi, api, synth, n_gpus):
    """End to end from a FASTQ file on disk, host decompression and parsing included: trew_multi_process_file (the
    reference's read_fastq_thread restated + packing + H2D + kernels on every GPU of the group) followed by
    trew_multi_finish; and the drop-in `trew` binary itself on the same files (process start, context creation and the
    report included -- what a user of the command line sees)."""
    import gzip
    n = 2_000_000
    tmp = tempfile.mkdtemp(prefix="trew_file_")
    out = {"gpus": n_gpus}
    try:
        plain = os.path.join(tmp, "r.fastq")
        with open(plain, "wb") as f:
            for i in range(0, n, 250_000):
                mat = synth.config_short(31 + i, 250_000, READ_LEN, telomeric=SYNTH["tel_ppm"] / 1e6,
                                         half_telomeric=SYNTH["half_ppm"] / 1e6, n_rate=SYNTH["n_ppm"] / 1e6,
                                         sub=SYNTH["sub_ppm"] / 1e6)
                f.write(synth.fastq_matrix_bytes(mat))
        gz = plain + ".gz"
        with open(plain, "rb") as src, gzip.open(gz, "wb", compresslevel=1) as dst:
            shutil.copyfileobj(src, dst, 1 << 24)
        bgz = plain + ".bgz"
        synth.bgzf_write(plain, bgz)
        env = dict(os.environ, TREW_DEVICES="all")
        for name, path in (("plain_fastq", plain), ("fastq_gz", gz), ("fastq_bgzf", bgz)):
            best = None
            for _ in range(2):
                multi.reset()
                t0 = time.perf_counter()
                multi.process_file(path)
                multi.finish_view()
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            t0 = time.perf_counter()
            subprocess.run([api.CLI_PATH, "short", "5", "32", path], check=True, stdout=subprocess.DEVNULL, env=env)
            cli_s = time.perf_counter() - t0
            out[name] = {"value": n * READ_LEN / best / 1e9, "unit": "Gbases/s", "reads": n, "file_bytes": os.path.getsize(path),
                         "trew_cli": {"wall_s": cli_s, "value": n * READ_LEN / cli_s / 1e9, "unit": "Gbases/s"}}
        out["note"] = ("one file: a plain gzip member is ONE DEFLATE stream (the reference reads it through one gzread); here all host threads "
                       "decode it together (speculative block starts, pinflate.cpp; this file is gzip -1, the worst case: more symbols per byte; "
                       "TREW_NO_PARALLEL_GZ=1 gives the one-core figure); BGZF (bgzip) members are inflated in parallel; plain FASTQ is bound by the newline index and the packer, both working "
                       "on the mapped file.  trew_cli = the `trew short 5 32 FILE` binary as a subprocess, wall clock: CUDA context creation "
                       "and pinned-buffer allocation (a fixed ~0.5-1 s per GPU) dominate at this file size")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return out


def cpu_baseline():
    cores = os.cpu_count() or 1
    if not reference_available():
        return {"value": None, "unit": "Gbases/s", "cores": cores, "kind": "reference", "sample": "oracle/_ref not built"}
    tmp = tempfile.mkdtemp(prefix="trew_cpu_")
    try:
        n = 120_000 * cores  # ~15-25 s of CPU work at ~0.8 Mbases per core-second
        p = os.path.join(tmp, "sample.fastq")
        write_sample_fastq(p, n)
        t = time_reference(p, cores)
        return {"value": n * READ_LEN / t / 1e9, "unit": "Gbases/s", "cores": cores, "kind": "reference",
                "sample": "%d reads of the same distribution (numpy generator) as plain FASTQ, `trew_ref short 5 32 -t %d -q 1024` "
                          "(unmodified reference sources + shim containers), wall clock %.1f s" % (n, cores, t)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of the headline figure; the e2e and configs figures time min(steps, 5) steps each")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=200_000_000, help="configs[1]: 200 M reads -- in total (strong) or per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): the 200 M reads are sharded over the GPUs; weak: every GPU holds --reads reads")
    ap.add_argument("--e2e-reads", type=int, default=8_000_000, help="reads per GPU and end-to-end step (host buffers)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--full-tables", action="store_true", help="time the steps with every table row copied to the host (no report filter)")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling figure beside the strong one")
    ap.add_argument("--no-shapes", action="store_true", help="skip the paired / long / 3-64 shapes (configs[2..4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the tables of the last timed step to DIR/{table,k,seq,count}.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the tables of --impl ours")
    # stdout carries exactly one JSON line (rank 0): native libraries that print there (NCCL's version banner)
    # are diverted to stderr for the duration of the run
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = run_reference_arm(args) if args.impl == "reference" else run_ours(args)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
