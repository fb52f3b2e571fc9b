#!/usr/bin/env python
"""bench.py — compaction throughput of the B200 path (and of the reference's CPU path, --impl reference).

One step = one whole compaction job: k pre-staged BlockBasedTable images (device resident) -> decode -> k-way merge
with the compaction-iterator rules -> BlockBasedTable output images.  Workload at every N: per GPU, the configuration
BASELINE.json's metric is quoted on (configs[1]: 8-way merge, 8 x 256 MiB synthetic sorted runs, 16 B keys / 32 B
values); ranks hold disjoint key ranges = independent sub-compactions (weak scaling), and after every step all-gather
the (smallest, largest) internal keys of their outputs over NCCL to stitch / assert the level's key order.

metric  : compaction MB/s of input KV bytes (sum over input entries of internal-key + value bytes), MB = 1e6 bytes
value   : device-resident inputs, CUDA-event time on the job stream, max over ranks
e2e     : same job through the C ABI with HOST (pinned) input images and host outputs, H2D + D2H inside the timed region
          (several jobs in flight, as concurrent background compactions are); e2e.single_job_ms: one job alone, uploaded whole;
          e2e.single_job_pipelined: one job alone as key-range sub-jobs whose inputs are uploaded in key order
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from toplingdb_b200.synth_workloads import BENCH_JOB, WORKLOADS  # noqa: E402  (no torch import: the reference arm needs none)


def source_sha16():
    """digest of the CUDA sources the library is built from (the ncu traffic file is stamped with it)"""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "toplingdb_b200", "csrc")
    for f in sorted(os.listdir(d)):
        h.update(f.encode())
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons of one GPU, sampled every ~2 ms from a thread.  NVML is initialised by the constructor (it takes
    longer than a whole timed region), sampling starts with start(), and summary() only counts the samples taken between
    mark_begin() and mark_end() -- the timed region(s)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        self.windows = []  # [begin, end] of the timed regions (perf_counter)
        self.nvml = None
        try:
            import pynvml as N
            N.nvmlInit()
            self.handle = N.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = N.nvmlDeviceGetMaxClockInfo(self.handle, N.NVML_CLOCK_SM)
            self.get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
            self.nvml = N
        except Exception:
            self.nvml = None

    def mark_begin(self):
        self.windows.append([time.perf_counter(), float("inf")])

    def mark_end(self):
        self.windows[-1][1] = time.perf_counter()

    def sample_nvml(self):
        N = self.nvml
        bits = [(0x8, 3), (0x40, 4), (0x20, 5), (0x4, 6)]  # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap -> row columns
        r = int(self.get_reasons(self.handle))
        row = [str(N.nvmlDeviceGetClockInfo(self.handle, N.NVML_CLOCK_SM)), str(self.max_mhz), "0", "", "", "", ""]
        for bit, col in bits:
            row[col] = "Active" if r & bit else "Not Active"
        return row

    def run(self):
        if self.nvml is not None:
            while not self.stop_flag:
                try:
                    self.rows.append((time.perf_counter(), self.sample_nvml()))
                except Exception:
                    break
                time.sleep(0.002)
            if self.rows:
                return
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append((time.perf_counter(), [x.strip() for x in out.split(",")]))
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        wins = self.windows or [[0.0, float("inf")]]
        rows = [r for t, r in self.rows if any(lo <= t <= hi for lo, hi in wins)]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows if len(r) > 3 + i)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "samples": len(rows), "sm_min_mhz": min(sm) if sm else None, "timed_regions": len(self.windows)}


DUMP_SAMPLE_BYTES = 4 << 20  # output bytes kept by --dump-outputs per run: 16 MiB of values + 32 MiB of positions


def dump_outputs(jobs, out_dir, rank, world):
    """--dump-outputs: what a caller of the timed path receives from its last step, as .npy files that two builds can be compared on.
    file_meta (float64, one row per output file of every job): the job's index, then the numeric fields of FileMeta in header order;
    output_keys (float32 [files, 2, 64]): the bytes of the smallest and the largest internal key (zero padded);
    job_stats (float64, one row per job): the counters of JobStats (its timings are left out: they change from run to run);
    output_bytes (float32) at output_byte_positions (float64): the bytes of the output tables laid end to end, all of them or a
    seeded sample of DUMP_SAMPLE_BYTES positions, so that the whole dump stays under 64 MB."""
    import numpy as np
    import torch
    from toplingdb_b200.native import FileMeta, JobStats
    if world > 1:
        out_dir = os.path.join(out_dir, f"rank{rank}")
    os.makedirs(out_dir, exist_ok=True)
    files = [(jx, j, i, j.output_meta(i)) for jx, j in enumerate(jobs) for i in range(j.output_count())]
    meta_fields = [n for n, _ in FileMeta._fields_ if not n.endswith("_ikey")]
    meta = [[jx] + [getattr(m, n) for n in meta_fields] for jx, _, _, m in files]
    keys = np.zeros((len(files), 2, 64), dtype=np.float32)
    for f, (_, _, _, m) in enumerate(files):
        keys[f, 0] = list(m.smallest_ikey)
        keys[f, 1] = list(m.largest_ikey)
        keys[f, 0, min(m.smallest_ikey_len, 64):] = 0
        keys[f, 1, min(m.largest_ikey_len, 64):] = 0
    stat_fields = [n for n, _ in JobStats._fields_ if not n.endswith("_us")]
    stats = [[getattr(s, n) for n in stat_fields] for s in (j.stats() for j in jobs)]
    sizes = np.array([m.file_size for _, _, _, m in files], dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    n_sample = DUMP_SAMPLE_BYTES // world
    if starts[-1] <= n_sample:
        pos = np.arange(starts[-1], dtype=np.int64)
    else:
        pos = np.sort(np.random.default_rng(0).integers(0, starts[-1], n_sample))
    vals = []
    for f, (_, j, i, m) in enumerate(files):
        lo, hi = np.searchsorted(pos, [starts[f], starts[f + 1]])
        img = torch.empty(m.file_size, dtype=torch.uint8, device=torch.device("cuda", j.params.device))
        j.output_read_into(i, img)
        vals.append(img[torch.from_numpy(pos[lo:hi] - starts[f]).to(img.device)].cpu().numpy())
    np.save(os.path.join(out_dir, "file_meta.npy"), np.array(meta, dtype=np.float64).reshape(len(files), 1 + len(meta_fields)))
    np.save(os.path.join(out_dir, "output_keys.npy"), keys)
    np.save(os.path.join(out_dir, "job_stats.npy"), np.array(stats, dtype=np.float64))
    np.save(os.path.join(out_dir, "output_bytes.npy"), np.concatenate(vals or [np.zeros(0, np.uint8)]).astype(np.float32))
    np.save(os.path.join(out_dir, "output_byte_positions.npy"), pos.astype(np.float64))


def reference_arm(args, rank, world):
    """The reference's own CPU ProcessKeyValueCompaction (oracle/_ref = the unmodified reference compiled here; else the
    CPU oracle port), all host threads, on a bounded sample of the same workload."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cpu_baseline as CB
    w = WORKLOADS[args.workload]
    cores = CB.usable_cores()
    # one process per usable host core (CPU affinity capped by the cgroup quota), each compacting its own key range of 64 MiB
    # raw KV: long enough to span several scheduler quota periods, so that a burst above the quota does not flatter the number
    sample = max(args.sample_mb << 20, cores * (64 << 20))
    res = []
    for _ in range(max(1, args.warmup > 0) + args.steps):
        res.append(CB.run_sample(w, sample_bytes=sample, threads=cores))
    res = res[1:] if len(res) > args.steps else res
    mbps = statistics.mean(r["mbps"] for r in res)
    # the same cores used the other way the reference can: ONE job split by max_subcompactions (threads inside one CompactionJob)
    sub = CB.run_subcompactions(w, sample_bytes=sample, threads=cores)
    line = {"impl": "reference", "metric": "compaction_input_kv_MB_per_s", "value": mbps, "unit": "MB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": statistics.mean(r["seconds"] for r in res) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": w["desc"], "sample": res[0]["sample"]},
            "cpu_baseline": {"value": mbps, "unit": "MB/s", "cores": cores, "kind": res[0]["kind"], "sample": res[0]["sample"]},
            "e2e": {"value": mbps, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if sub:
        line["one_job_max_subcompactions"] = {"value": round(sub["mbps"], 1), "unit": "MB/s", "max_subcompactions": sub["max_subcompactions"],
                                              "sub_compactions_formed": sub["sub_compactions_formed"], "sample": sub["sample"]}
    print(json.dumps(line))


def plugin_arm(args, rank):
    """bench.py --impl plugin: the CompactionExecutor plugin path of the reference DB (oracle/_ref/ref_compact_b200) on one job, with the
    stock binary's local compaction beside it.  Wall time of the executor's Execute (CompactionJobStats.elapsed_micros)."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cpu_baseline as CB
    w = WORKLOADS[args.workload]
    r = CB.run_plugin_sample(w, sample_bytes=max(args.sample_mb, 512) << 20)
    if r is None:
        print(json.dumps({"impl": "plugin", "unavailable": "oracle/_ref/ref_compact_b200 is not built"}))
        return
    line = {"impl": "plugin", "metric": "compaction_input_kv_MB_per_s", "value": round(r["plugin"]["mbps"], 1), "unit": "MB/s", "n_gpus": 1,
            "ms_per_step": round(r["plugin"]["seconds"] * 1e3, 2), "higher_is_better": True, "dtype": "u8", "data": "synthetic",
            "config": {"workload": w["desc"], "sample": r["sample"]},
            "executor": r["plugin"]["executor"], "remote_compact_read_bytes": r["plugin"]["remote_compact_read_bytes"],
            "local_cpu_compaction": {"value": round(r["local"]["mbps"], 1), "unit": "MB/s", "ms": round(r["local"]["seconds"] * 1e3, 2)},
            "plugin_4_ranges": {"value": round(r["plugin_4_ranges"]["mbps"], 1), "unit": "MB/s", "ms": round(r["plugin_4_ranges"]["seconds"] * 1e3, 2)},
            "speedup_vs_local": round(r["plugin"]["mbps"] / r["local"]["mbps"], 2)}
    print(json.dumps(line))


def concurrent_jobs_arm(args, w, rank, world, local, numa_info):
    """BASELINE.json configs[4]: J independent sub-compactions per GPU, all in flight at once (one host thread and one stream pair per
    job), ranks hold disjoint key ranges.  A step = every job of the rank run once; device time between two events that bracket the
    step (all streams drained on both sides), max over ranks."""
    import threading
    import torch
    import torch.distributed as dist
    import toplingdb_b200 as T
    from toplingdb_b200 import synth
    J, base = w["jobs"], w["base"]
    common = dict(device=local, bottommost_level=w["bottommost"], **BENCH_JOB)
    sets, kv_bytes, in_bytes = [], 0, 0
    for jx in range(J):
        images, kv = synth.stage_bench_inputs(base, rank=rank * J + jx, scale=args.scale, device_index=local)
        sets.append(images)
        kv_bytes += kv
        in_bytes += sum(int(t.numel()) for t in images)
    jobs = []
    for jx, images in enumerate(sets):
        job = T.CompactionJob(output_mem="device", profile=1 if jx == 0 else 0, **common)
        for i, img in enumerate(images):
            job.add_input(img, level=0, file_number=100 + i)
        jobs.append(job)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def run_all(js):
        errs = []

        def one(j):
            try:
                j.run()
                _ = j.stats().num_output_records
            except Exception as e:  # noqa: BLE001
                errs.append(e)
        ths = [threading.Thread(target=one, args=(j,)) for j in js]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        if errs:
            raise errs[0]

    sampler = ClockSampler(local)
    sampler.start()  # (samples outside the timed regions are dropped by summary())
    for _ in range(args.warmup):
        run_all(jobs)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    sampler.mark_begin()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run_all(jobs)
    torch.cuda.synchronize()
    ev1.record()
    barrier()
    sampler.mark_end()
    wall_s = (time.perf_counter() - t0) / args.steps
    step_s = ev0.elapsed_time(ev1) / 1e3 / args.steps
    out_bytes = sum(j.output_meta(i).file_size for j in jobs for i in range(j.output_count()))
    nout = sum(j.output_count() for j in jobs)
    launches = sum(j.stats().kernel_launches for j in jobs)
    kern = [{"name": n, "us": round(us, 1)} for n, us in jobs[0].kernel_times()]
    if args.dump_outputs:
        dump_outputs(jobs, args.dump_outputs, rank, world)
    if world > 1:
        tt = torch.tensor([step_s, wall_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        step_s, wall_s = tt.tolist()
    value = world * kv_bytes / step_s / 1e6
    pk, pk_src = peaks()
    # whole-step figure against the HBM roofline: every input byte read once + every output byte written once
    ach = (in_bytes + out_bytes) / step_s / 1e9
    roofline = {"bound": "hbm", "kernel": "whole step (8 jobs in flight)", "achieved": round(ach, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": round(ach / pk["hbm_gbs"], 4), "traffic": None, "peak_source": pk_src}
    e2e = None
    if not args.no_e2e:
        host_sets = [[t.cpu().pin_memory() for t in images] for images in sets]
        for j in jobs:
            j.close()
        del sets
        torch.cuda.empty_cache()
        ejs = []
        for images in host_sets:
            ej = T.CompactionJob(output_mem="host", **common)
            for i, img in enumerate(images):
                ej.add_input(img, level=0, file_number=100 + i)
            ejs.append(ej)
        run_all(ejs)
        barrier()
        sampler.mark_begin()
        t0 = time.perf_counter()
        reps = max(2, min(args.steps, 4))
        for _ in range(reps):
            run_all(ejs)
        barrier()
        sampler.mark_end()
        es = (time.perf_counter() - t0) / reps
        if world > 1:
            tt = torch.tensor([es], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            es = tt.item()
        e2e = {"value": round(world * kv_bytes / es / 1e6, 1), "unit": "MB/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": out_bytes,
               "ms_per_step": round(es * 1e3, 2), "steps": reps, "jobs_in_flight": J}
        for ej in ejs:
            ej.close()
    sampler.stop_flag = True
    if rank == 0:
        line = {"metric": "compaction_input_kv_MB_per_s", "value": round(value, 1), "unit": "MB/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(step_s * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic",
                "config": {"workload": w["desc"] + (f" (scale {args.scale})" if args.scale != 1.0 else ""), "jobs_per_gpu": J, "k": w["k"],
                           "input_kv_bytes_per_gpu": kv_bytes, "input_sst_bytes_per_gpu": in_bytes, "output_files_per_gpu": nout,
                           "output_sst_bytes_per_gpu": out_bytes, "l2_policy": "inputs (2.2 GB per GPU) >> 126 MB L2",
                           "parallelism": f"{world} GPUs x {J} independent sub-compactions", "numa": numa_info},
                "wall_ms_per_step": round(wall_s * 1e3, 3), "e2e": e2e, "gpu_launches": int(launches) * args.steps, "roofline": roofline,
                "kernels_of_job0_while_8_run": kern, "cpu_baseline": None, "clocks": sampler.summary()}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the per-run size (debug only; invalidates the number)")
    ap.add_argument("--sample-mb", type=int, default=192, help="raw KV MiB of the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-depth", type=int, default=4, help="compaction jobs in flight in the end-to-end measurement")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--pipeline-ranges", type=int, default=8, help="key ranges of the pipelined single-job measurement (e2e.single_job_pipelined)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return reference_arm(args, rank, world)
    if args.impl == "plugin":
        return plugin_arm(args, rank)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import toplingdb_b200 as T
    from toplingdb_b200 import sharding, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the compaction path has no CPU implementation)")
    torch.cuda.set_device(local)
    # host buffers next to the GPU: CPU affinity + memory policy of this rank go to the GPU's NUMA node before anything is pinned
    from toplingdb_b200 import numa
    numa_info = numa.bind_to_gpu_node(local) if not args.no_numa else {"gpu": local, "node": None, "cpus": None, "mempolicy": False}
    if world > 1:
        # the bench prints exactly one JSON line on stdout: keep NCCL's own banner / logs on stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    w = WORKLOADS[args.workload]
    if w.get("jobs", 1) > 1:
        return concurrent_jobs_arm(args, w, rank, world, local, numa_info)
    # ranks hold disjoint, ordered key ranges = independent sub-compactions; tests/test_gpu_fullsize.py stages the same job (rank 0) and
    # compares every output byte with the CPU oracle
    images, kv_bytes = synth.stage_bench_inputs(args.workload, rank=rank, scale=args.scale, device_index=local)
    in_bytes = sum(int(t.numel()) for t in images)
    common = dict(device=local, bottommost_level=w["bottommost"], **BENCH_JOB)
    job = T.CompactionJob(output_mem="device", profile=1, **common)
    for i, img in enumerate(images):
        job.add_input(img, level=0, file_number=100 + i)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def boundary_exchange():
        """the path's one collective: all-gather of each rank's 64-byte output boundary record + non-overlap check"""
        if world > 1:
            sharding.exchange_boundaries(sharding.job_boundary(job), device=torch.device("cuda", local))

    sampler = ClockSampler(local)
    sampler.start()  # (samples outside the timed regions are dropped by summary())
    for _ in range(args.warmup):
        job.run()
        boundary_exchange()
    barrier()
    dev_us, ktimes = [], {}
    sampler.mark_begin()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        job.run()
        boundary_exchange()
        st = job.stats()
        dev_us.append(st.total_us)
        for name, us in job.kernel_times():
            ktimes.setdefault(name, []).append(us)
    barrier()
    sampler.mark_end()
    wall = time.perf_counter() - t0
    st = job.stats()
    nout = job.output_count()
    out_bytes = sum(job.output_meta(i).file_size for i in range(nout))
    out_data = sum(job.output_meta(i).data_size for i in range(nout))
    launches = st.kernel_launches
    # timing: device time per step, max over ranks
    step_s = sum(dev_us) / 1e6 / args.steps
    wall_s = wall / args.steps
    if world > 1:
        tt = torch.tensor([step_s, wall_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        step_s, wall_s = tt.tolist()
    value = world * kv_bytes / step_s / 1e6

    # untimed checks: the outputs of the last step hash to the digest the CPU oracle produced for this very job (committed by
    # tools/make_bench_digests.py, re-derived by tests/test_gpu_fullsize.py on every GPU test run); entry conservation; file order
    digest = synth.outputs_digest(job)
    dkey = f"{args.workload}:rank{rank}:scale{args.scale}"
    want_digest = None
    try:
        want_digest = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_digests.json"))).get(dkey)
    except Exception:
        pass
    if want_digest is not None and want_digest != digest:
        raise SystemExit(f"bench outputs differ from the oracle's ({dkey}): {digest} != {want_digest}")
    if w["overlap"] == 0 and w["del_frac"] == 0:
        assert st.num_output_records == st.num_input_records, (st.num_output_records, st.num_input_records)
    prev = None
    for i in range(nout):
        m = job.output_meta(i)
        a, b = bytes(m.smallest_ikey[:16]), bytes(m.largest_ikey[:16])
        assert a <= b and (prev is None or prev < a), "output files out of order"
        prev = b
    if args.dump_outputs:
        dump_outputs([job], args.dump_outputs, rank, world)

    # per-kernel roofline on the dominant kernel group
    pk, pk_src = peaks()
    n_in, n_out = st.num_input_records, st.num_output_records
    in_data = in_bytes  # data blocks dominate the image; index/tail < 1.5 %
    val_out = st.total_input_raw_value_bytes if n_out == n_in else int(st.total_input_raw_value_bytes * n_out / max(1, n_in))
    # Algorithmic bytes per launch, SURVEY.md 8(d): every input (ikey + value) byte read once + every surviving output byte
    # written once -- decode: SST file bytes read + raw KV bytes written; merge: raw KV read + surviving raw KV written
    # (112 B per input entry on cfg2); encode: raw KV bytes read + SST file bytes written.  `moved_bytes` is what the kernel
    # really has to move in this design (values stay in the input image until the emit kernel: 36-byte columns instead).
    kv_in = st.total_input_raw_key_bytes + st.total_input_raw_value_bytes
    kv_out = kv_in if n_out == n_in else int(kv_in * n_out / max(1, n_in))
    algo = {
        "decode.blocks": in_data + kv_in,
        "merge.tiles": kv_in + kv_out,
        "encode.emit": kv_out + out_data,
    }
    moved = {
        "decode.blocks": in_data + 36 * n_in,
        "merge.tiles": 36 * n_in + 36 * n_out,
        "encode.sizes": 28 * n_out + 5 * n_out,
        "encode.tables": 9 * n_out + 6 * n_out,
        "encode.emit": 36 * n_out + val_out + out_data,
    }
    kern = []
    for name, xs in ktimes.items():
        us = statistics.mean(xs)
        ab, mb = algo.get(name, 0), moved.get(name, 0)
        kern.append({"name": name, "us": round(us, 1), "algo_bytes": ab, "gbs": round(ab / us / 1e3, 1) if us > 0 else None,
                     "moved_bytes": mb, "moved_gbs": round(mb / us / 1e3, 1) if us > 0 else None})
    kern.sort(key=lambda x: -x["us"])
    # groups whose name starts with '~' run on the job's side stream, overlapped with the neighbouring group of the main stream
    # (their time is not part of the step's critical path): they are listed, but never the dominant kernel
    dom = next((x for x in kern if not x["name"].startswith("~")), None)
    # DRAM bytes of the dominant kernel from the ncu capture of THIS library build (profiles/ncu_traffic.json carries the sha256 of the
    # libb200c.so it was taken from; a capture of another build is not reported)
    traffic = None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if dom and os.path.exists(tp):
        import hashlib
        tj = json.load(open(tp))
        lib_sha = hashlib.sha256(open(os.path.join(ROOT, "toplingdb_b200", "libb200c.so"), "rb").read()).hexdigest()[:16]
        if tj.get("lib_source_sha16") in (None, source_sha16()) or tj.get("lib_sha16") == lib_sha:
            traffic = tj.get(dom["name"])
    roofline = None
    if dom:
        ach = dom["algo_bytes"] / dom["us"] / 1e3
        roofline = {"bound": "hbm", "kernel": dom["name"], "achieved": round(ach, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": round(ach / pk["hbm_gbs"], 4), "traffic": traffic, "peak_source": pk_src,
                    "algo_bytes_per_launch": dom["algo_bytes"], "avg_us": dom["us"],
                    "convention": "SURVEY 8(d): raw KV / SST bytes in + out of the stage", "moved_bytes_per_launch": dom["moved_bytes"]}
        mt = next((x for x in kern if x["name"] == "merge.tiles"), None)
        if mt:  # the kernel BASELINE.json's 40 % target is quoted on
            roofline["merge"] = {"achieved": mt["gbs"], "frac": round(mt["gbs"] / pk["hbm_gbs"], 4), "avg_us": mt["us"],
                                 "algo_bytes_per_launch": mt["algo_bytes"], "moved_gbs": mt["moved_gbs"]}

    # e2e through the C ABI with host buffers (pinned), H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        host_imgs = [t.cpu().pin_memory() for t in images]
        job.close()
        del images
        torch.cuda.empty_cache()
        # Several jobs in flight (one host thread per job, each job on its own stream): the upload of one job overlaps the download
        # of the other, as concurrent background compactions do (max_background_compactions > 1).  Every step still does
        # its own H2D of the inputs and D2H of the outputs inside the timed region.
        import threading
        depth = max(1, args.e2e_depth)
        ejs = [T.CompactionJob(output_mem="host", **common) for _ in range(depth)]
        for ej in ejs:
            for i, img in enumerate(host_imgs):
                ej.add_input(img, level=0, file_number=100 + i)
            ej.run()
        barrier()
        t0 = time.perf_counter()  # one job alone: the latency a single compaction sees
        ejs[0].run()
        _ = ejs[0].stats().num_output_records
        barrier()
        single_s = time.perf_counter() - t0
        per_thread = max(2, (min(args.steps, 6) + depth - 1) // depth)  # every job runs at least twice in the timed region
        esteps = per_thread * depth
        errs = []

        def worker(ej):
            try:
                for _ in range(per_thread):
                    ej.run()
                    _ = ej.stats().num_output_records  # the result the caller reads
            except Exception as e:  # noqa: BLE001
                errs.append(e)

        barrier()
        sampler.mark_begin()
        t0 = time.perf_counter()
        ths = [threading.Thread(target=worker, args=(ej,)) for ej in ejs]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        barrier()
        sampler.mark_end()
        es = (time.perf_counter() - t0) / esteps
        if errs:
            raise errs[0]
        if world > 1:
            tt = torch.tensor([es], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            es = tt.item()
        e2e = {"value": round(world * kv_bytes / es / 1e6, 1), "unit": "MB/s", "h2d_bytes_per_step": in_bytes,
               "d2h_bytes_per_step": out_bytes, "ms_per_step": round(es * 1e3, 2), "steps": esteps, "jobs_in_flight": depth,
               "single_job_ms": round(single_s * 1e3, 2)}
        for ej in ejs:
            ej.close()
        del ejs
        # ONE job alone, pipelined over its own PCIe link: the inputs go up in key order and the job runs as key-range sub-jobs
        # (b200c_job_plan_ranges / b200c_job_upload_by_ranges / b200c_job_create_sub), each of which starts -- and downloads its
        # outputs -- as soon as its own blocks have arrived.  Its outputs are those of the ranges (what the reference writes with
        # max_subcompactions > 1), checked per range in tests/test_gpu_subjobs.py; here: entry conservation.
        try:
            def pipelined_once():
                parent = T.CompactionJob(output_mem="host", **common)
                for i, img in enumerate(host_imgs):
                    parent.add_input(img, level=0, file_number=100 + i, deferred=True)
                bounds = parent.plan_ranges(args.pipeline_ranges, min_range_bytes=BENCH_JOB["max_output_file_size"])
                parent.upload_by_ranges(bounds)
                rng = list(zip([None] + bounds, bounds + [None]))
                subs = [parent.sub_job(range_start=a, range_end=b, first_file_number=1000 * (x + 1)) for x, (a, b) in enumerate(rng)]
                perr = []

                def go(sj):
                    try:
                        sj.run()
                    except Exception as e:  # noqa: BLE001
                        perr.append(e)
                pth = [threading.Thread(target=go, args=(sj,)) for sj in subs]
                for th in pth:
                    th.start()
                for th in pth:
                    th.join()
                if perr:
                    raise perr[0]
                n_in = sum(sj.stats().num_input_records for sj in subs)
                n_files = sum(sj.output_count() for sj in subs)
                for sj in subs:
                    sj.close()
                parent.close()
                return len(rng), n_in, n_files
            pipelined_once()  # buffers of the sub-jobs come from the library's cache afterwards, as for the other numbers
            barrier()
            t0 = time.perf_counter()
            nr, n_in_p, nf_p = pipelined_once()
            barrier()
            e2e["single_job_pipelined"] = {"ms": round((time.perf_counter() - t0) * 1e3, 2), "key_ranges": nr, "output_files": nf_p,
                                           "input_records": n_in_p}
            assert n_in_p == st.num_input_records, (n_in_p, st.num_input_records)
        except Exception as e:  # noqa: BLE001
            e2e["single_job_pipelined"] = {"error": repr(e)[:200]}

    sampler.stop_flag = True
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import cpu_baseline as CB
        r = CB.run_sample(w, sample_bytes=min(args.sample_mb, 128) << 20, threads=1)
        cpu = {"value": round(r["mbps"], 1), "unit": "MB/s", "cores": 1, "kind": r["kind"], "sample": r["sample"]}

    if rank == 0:
        line = {"metric": "compaction_input_kv_MB_per_s", "value": round(value, 1), "unit": "MB/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(step_s * 1e3, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": {"workload": w["desc"] + (f" (scale {args.scale})" if args.scale != 1.0 else ""), "k": w["k"],
                           "entries_per_gpu": n_in, "input_kv_bytes_per_gpu": kv_bytes, "input_sst_bytes_per_gpu": in_bytes,
                           "output_files_per_gpu": nout, "output_sst_bytes_per_gpu": out_bytes, "l2_policy": "inputs (2.2 GB) >> 126 MB L2",
                           "parallelism": f"{world} independent sub-compactions, 1 per GPU" if world > 1 else "1 GPU", "numa": numa_info},
                "wall_ms_per_step": round(wall_s * 1e3, 3), "e2e": e2e, "gpu_launches": int(launches) * args.steps, "roofline": roofline,
                "kernels": kern, "cpu_baseline": cpu, "clocks": sampler.summary(),
                "output_digest": {"sha256": digest, "oracle": want_digest, "matches_oracle": (want_digest == digest) if want_digest else None},
                "stage_us": {"decode": round(st.decode_us, 1), "merge": round(st.merge_us, 1), "encode": round(st.encode_us, 1)}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
