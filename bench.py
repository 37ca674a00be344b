#!/usr/bin/env python
"""bench.py -- SSB Q4.1 (scan -> 4-way hash join -> group-by) rows/sec on N B200s, beside the CPU oracle.

Contract (see DESIGN.md "Measurement"):
  python bench.py --gpus N --steps K --warmup W          (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W   (CPU arm: the oracle on host cores)
prints ONE JSON line on rank 0.

A "step" is one pass of the hot path over one batch: the whole lineorder shard of the rank (SF100 = 600 M
rows per GPU, weak scaling) goes through the fused fragment (scan -> probe x4 -> aggregate), the partial
group-by states are pulled, and for N > 1 gathered over NCCL and merged by a final GPU aggregate on rank 0.
  value : rows/s with the fact columns already resident in HBM when the timed region starts
  e2e   : the same through the C-ABI with HOST (pinned) column buffers, H2D inside the timed region
The inputs (14.4 GB of fact columns per GPU) are far larger than the 126 MB L2, so no L2 flush is needed
between timed iterations (config.l2: "inputs >> L2").
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

ALGO_BYTES_PER_ROW = 24  # SURVEY.md section 8d: 6 int32 fact columns


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gpu", choices=["gpu", "reference"])
    ap.add_argument("--workload", default="q41", choices=["q41", "groupby", "q3", "q95"],
                    help="q41: SSB SF100 Q4.1 (BASELINE.json's metric; the default).  groupby: BASELINE.json config 5, 1e9 rows / 1e8 "
                         "distinct int64 keys, SUM + COUNT, on one B200 (N > 1: one independent key range per GPU, no exchange).  "
                         "q3: BASELINE.json config 3, TPC-H Q3 with the NCCL hash shuffle (tools/q3_distributed.py; --sf = TPC-H scale).  "
                         "q95: BASELINE.json config 4, the TPC-DS Q95 shape (tools/q95_distributed.py; --sf = TPC-DS scale, default 1000 / 8 per GPU)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="q41 with N > 1: weak = --sf per GPU (default), strong = --sf split over the N GPUs")
    ap.add_argument("--groupby-rows", type=int, default=1_000_000_000)
    ap.add_argument("--groupby-keys", type=int, default=100_000_000)
    ap.add_argument("--sf", type=float, default=100.0, help="SSB scale factor per GPU (weak scaling)")
    ap.add_argument("--rows", type=int, default=0, help="override fact rows per GPU")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-morsel-rows", type=int, default=1 << 22,
                    help="e2e: the host columns are pushed in morsels of this many rows (measured: 4 M-row morsels 170.6 ms per 600 M rows, "
                         "one 600 M-row batch 197 ms; tools/e2e_batches.py)")
    ap.add_argument("--no-operator-e2e", action="store_true", help="skip e2e.operator_api (the C++ operator path, starrocks_b200/host/bench)")
    ap.add_argument("--cpu-sample-rows", type=int, default=0, help="rows of the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--merge", choices=["allreduce", "gather"], default="allreduce",
                    help="N>1 merge of the partial aggregates: in-place all-reduce of the dense slot arrays (SURVEY 8e) or "
                         "gather of partial rows to rank 0 + final aggregate (the reference plan's UNPARTITIONED exchange)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="q41 GPU arm: after the timed steps, write the result columns of the last timed step as DIR/<name>.npy "
                         "(float64, rows sorted by group key) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "q41" or args.impl != "gpu"):
        ap.error("--dump-outputs is implemented for the q41 workload of the GPU arm")
    return args


# ---------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled through NVML from a background thread (about 1 kHz: the timed region of the
    default run is ~20 ms, far shorter than one `nvidia-smi -lms` period).  Started before the warm-up; only the samples
    taken between mark_begin() and mark_end() -- the timed region -- are reported (`window: "timed"`); if the region was
    too short to catch any, the samples of the warm-up + timed window are reported and `window` says so."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake"}

    def __init__(self, device_index):
        self.idx = device_index
        self.samples = []   # (t, sm_mhz, reason bits)
        self.t0 = self.t1 = None
        self.thread = None
        self.smax = None
        self.err = None
        self._stop = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.idx
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.smax = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        except Exception as e:  # noqa: BLE001
            self.err = f"NVML unavailable: {e}"
            return

        def loop():
            while not self._stop:
                try:
                    self.samples.append((time.perf_counter(), pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), int(get_reasons(h))))
                except Exception as e:  # noqa: BLE001
                    self.err = str(e)
                    return
                time.sleep(0.001)
        import threading
        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        self._stop = True
        if self.thread is not None:
            self.thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.smax, "reasons": [self.err or "no samples"], "samples": 0}
        timed = [x for x in self.samples if self.t0 is not None and self.t1 is not None and self.t0 <= x[0] <= self.t1]
        window = "timed"
        if not timed:
            timed, window = self.samples, "warm-up + timed (timed region shorter than one sample period)"
        bits = 0
        for _, _, r in timed:
            bits |= r
        return {"sm_mhz": statistics.median(x[1] for x in timed), "sm_min_mhz": min(x[1] for x in timed), "sm_max_mhz": self.smax,
                "reasons": sorted(nm for b, nm in self.REASONS.items() if bits & b), "samples": len(timed), "window": window,
                "source": "NVML nvmlDeviceGetClockInfo / CurrentClocksEventReasons, 1 ms period"}


# ---------------------------------------------------------------------------------------------------
# data
# ---------------------------------------------------------------------------------------------------
def gen_lineorder_device(torch, dev, n, sz, seed):
    """SSB lineorder columns on the device (same distributions as ssb.gen_lineorder)."""
    from starrocks_b200 import ssb
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    datekey = torch.from_numpy(ssb.gen_dates()["d_datekey"]).to(dev)

    def ri(lo, hi):
        return torch.randint(lo, hi, (n,), dtype=torch.int32, device=dev, generator=g)
    cols = {}
    idx = torch.randint(0, datekey.numel(), (n,), dtype=torch.int64, device=dev, generator=g)
    cols["lo_orderdate"] = datekey[idx].contiguous()
    del idx
    cols["lo_custkey"] = ri(1, sz["customer"] + 1)
    cols["lo_suppkey"] = ri(1, sz["supplier"] + 1)
    cols["lo_partkey"] = ri(1, sz["part"] + 1)
    cols["lo_revenue"] = ri(81_000, 10_400_001)
    cols["lo_supplycost"] = ri(54_000, 125_001)
    return cols


def gen_lineorder_host(n, sz, seed):
    import torch
    from starrocks_b200 import ssb
    g = torch.Generator()
    g.manual_seed(seed)
    datekey = torch.from_numpy(ssb.gen_dates()["d_datekey"])

    def ri(lo, hi):
        return torch.randint(lo, hi, (n,), dtype=torch.int32, generator=g).numpy()
    cols = {"lo_orderdate": datekey[torch.randint(0, datekey.numel(), (n,), generator=g)].numpy().copy()}
    cols["lo_custkey"] = ri(1, sz["customer"] + 1)
    cols["lo_suppkey"] = ri(1, sz["supplier"] + 1)
    cols["lo_partkey"] = ri(1, sz["part"] + 1)
    cols["lo_revenue"] = ri(81_000, 10_400_001)
    cols["lo_supplycost"] = ri(54_000, 125_001)
    return cols


def host_cores():
    """threads the CPU arm can really run at once: the scheduler affinity, capped by the cgroup CPU quota (a 1-GPU lease may
    see all 128 cores in its affinity mask and still be throttled to a fraction of them: the same CPU arm ran 0.65 and
    3.5 G rows/s on two `128-core` boxes in round 1).  -> (threads to use, {"affinity": .., "cgroup_quota_cpus": ..})"""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]              # cgroup v2
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:                                                                     # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    eff = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return eff, {"affinity": aff, "cgroup_quota_cpus": quota}


def measured_peak():
    try:
        m = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(m["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def known_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return t
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU implementation of the path = the oracle (the BE cannot be built here)
# ---------------------------------------------------------------------------------------------------
def pcie_bytes_in_place(n, plan, width=4, n_cols=6, sector=64):
    """Bytes the fragment kernels fetch from pinned host memory for one in-place push: column k (in plan order) is read
    only for rows that survived the scan predicate and joins < k, in 64-byte bus blocks (the granularity measured with
    scripts/pcie_stride.cu); with uniformly distributed survivors of density d a block of 64/width rows is touched with
    probability 1-(1-d)^(64/width).  The aggregate input columns are read at the density left after the last join; the
    key of the streamed join whose payload is needed travels in the selection vector and is not read again."""
    per = sector // width
    d = float(plan.get("pred_rate", 1.0))
    total = 0.0
    rates = list(plan["pass_rate"])
    for k in range(n_cols):
        total += n * width * (1.0 - (1.0 - min(1.0, d)) ** per)
        if k < len(rates):
            d *= rates[k]
    return total


def oracle_run(oracle, ssb, abi, ojoins, cols, nrows, threads):
    chunk = abi.Chunk([(ssb.LO_SLOTS[nm], cols[nm][:nrows], None, abi.TYPE_INT) for nm in ssb.Q41_FACT_COLS])
    t0 = time.perf_counter()
    res, passed = oracle.fragment_run(abi.ScanDesc(), ojoins, ssb.q41_agg_desc(), chunk, num_threads=threads)
    return time.perf_counter() - t0, res, passed


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from starrocks_b200 import abi, ssb
    from oracle import oracle
    oracle.lib()
    sf = args.sf
    sz = ssb.sizes(sf)
    n_total = args.rows or sz["lineorder"]   # rows of one GPU's shard (weak) / of the whole table (strong)
    cores, cores_info = host_cores()
    dims = ssb.gen_dims(sf)
    ojoins, keep = ssb.build_dims(oracle, dims, ssb.dim_plans_q41())
    # bounded sample per step: sized from a probe run so that warmup + steps stay within a few minutes
    probe_rows = min(n_total, 8_000_000)
    cols = gen_lineorder_host(probe_rows, sz, ssb.SEED)
    dt, _, _ = oracle_run(oracle, ssb, abi, ojoins, cols, probe_rows, cores)
    rate = probe_rows / dt
    budget_s = 150.0 / max(1, args.steps + args.warmup)
    sample = int(min(n_total, max(4_000_000, rate * min(budget_s, 20.0))))
    if args.cpu_sample_rows:
        sample = min(n_total, args.cpu_sample_rows)
    cols = gen_lineorder_host(sample, sz, ssb.SEED)
    for _ in range(args.warmup):
        oracle_run(oracle, ssb, abi, ojoins, cols, sample, cores)
    times = []
    for _ in range(args.steps):
        dt, res, passed = oracle_run(oracle, ssb, abi, ojoins, cols, sample, cores)
        times.append(dt)
    total = sum(times)
    value = sample * args.steps / total
    line = {
        "impl": "reference", "metric": "rows/sec for SSB Q4.1 hash-join+agg", "value": value, "unit": "rows/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * total / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int32/int64", "data": "synthetic",
        "config": {"workload": f"SSB SF{sf:g} Q4.1 4-way hash join + group-by (scan->probe x4->aggregate)",
                   "fact_rows_per_gpu": n_total if args.scaling == "weak" else (n_total + max(1, args.gpus) - 1) // max(1, args.gpus),
                   "global_fact_rows": n_total * max(1, args.gpus) if args.scaling == "weak" else n_total,
                   "cpu_sample_rows_per_step": sample, "chunk_size": 4096,
                   "note": "StarRocks-semantics CPU restatement (oracle/), NOT the StarRocks BE binary: the BE cannot be built in this image"},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "kind": "port", "cores_detail": cores_info,
                         "sample": f"first {sample} lineorder rows of SF{sf:g} per step, {cores} pipeline drivers, 4096-row chunks"},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, result, names):
    """result columns (chunk_out_to_host form) -> out_dir/<names[slot]>.npy, float64 with NULL as NaN.  The rows are sorted
    by all columns, group keys first: the order in which the aggregate emits its groups is not part of the result."""
    from starrocks_b200.rows import gpu_rows
    rows = gpu_rows(result)
    os.makedirs(out_dir, exist_ok=True)
    for k, (slot, _, _, _) in enumerate(result):
        vals = [r[k] for r in rows]
        if any(v is not None and float(v) != v for v in vals):
            raise SystemExit(f"bench.py: column {names[slot]} is not exact in float64; refusing to dump a rounded value")
        np.save(os.path.join(out_dir, names[slot] + ".npy"), np.array([np.nan if v is None else v for v in vals], dtype=np.float64))


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from starrocks_b200 import abi, gpu, ssb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sf = args.sf
    sz = ssb.sizes(sf)
    n_global = args.rows or sz["lineorder"]
    # weak scaling: every GPU holds a whole --sf shard; strong scaling: the --sf fact table is split over the GPUs
    n = n_global if args.scaling == "weak" else (n_global + world - 1) // world
    # one explicit (non-default) stream shared by torch, NCCL and the library, so that torch CUDA events
    # bracket the library's kernels (the default stream's handle is 0 = "create your own" in sr_ctx_create)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = gpu.Context(local, stream=stream.cuda_stream)

    # ---- build side: 4 dimension scans + filters + join builds, replicated on every GPU (broadcast join) ----
    dims = ssb.gen_dims(sf)
    t0 = time.perf_counter()
    gjoins, gkeep = ssb.build_dims(gpu, dims, ssb.dim_plans_q41(), ctx=ctx)
    ctx.sync()
    build_ms = 1000.0 * (time.perf_counter() - t0)

    # ---- fact shard of this rank, resident in HBM ----
    cols = gen_lineorder_device(torch, dev, n, sz, ssb.SEED + 1000 * rank)
    torch.cuda.synchronize()
    dchunk = ssb.fact_chunk(cols, ssb.Q41_FACT_COLS, mem=abi.MEM_DEVICE)
    agg_desc = ssb.q41_agg_desc()
    frag = gpu.Fragment(ctx, abi.ScanDesc(), gjoins, agg_desc)

    # final (phase 2) aggregate on rank 0: SUM of the partial sums per (d_year, c_nation)
    final_desc = abi.make_agg_desc([ssb.D_YEAR, ssb.C_NATION], [abi.TYPE_INT, abi.TYPE_INT],
                                   fns=[(abi.AGG_SUM, abi.TYPE_BIGINT, ssb.OUT_SUM_REVENUE, [("col", ssb.OUT_SUM_REVENUE)]),
                                        (abi.AGG_SUM, abi.TYPE_BIGINT, ssb.OUT_SUM_SUPPLYCOST, [("col", ssb.OUT_SUM_SUPPLYCOST)])],
                                   ranges=[(1992, 1998), (0, 24)])
    final = gpu.Agg(ctx, final_desc) if world > 1 else None
    MAXG = 175

    def finish_step():
        """tail of a step: merge across ranks (N > 1) and bring the result to the host of rank 0"""
        if world > 1 and args.merge == "allreduce":
            from starrocks_b200.distributed import all_reduce_dense_state
            all_reduce_dense_state(frag.agg.dense_state(), dev)   # NCCL on the context's stream, in place
            frag.agg.finish()
            if rank != 0:
                return None
            return gpu.chunk_out_to_host(ctx, frag.agg.pull(mem=abi.MEM_HOST))
        frag.agg.finish()
        if world == 1:
            return gpu.chunk_out_to_host(ctx, frag.agg.pull(mem=abi.MEM_HOST))
        return step_tail(frag, final, ctx, gpu, abi, ssb, torch, dist, dev, world, rank, MAXG)

    def step(chunk):
        """one pass: push the shard, merge, pull the result to the host"""
        frag.reset()
        frag.push(chunk)
        return finish_step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    result = None
    for _ in range(max(args.warmup, 1)):
        result = step(dchunk)
    barrier()

    # ---- timed: value (HBM-resident inputs) ----
    launches0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    sampler.mark_begin()
    ev0.record(stream)
    pass_ms = [0.0, 0.0, 0.0]
    trace = [] if os.environ.get("SR_BENCH_TRACE") else None   # host-side phase timestamps (debug aid)
    for s in range(args.steps):
        # push() launches only the hot kernels of the path after the first batch (k_frag_stream,
        # k_frag_gather_join, k_frag_gather_agg -- or the single k_fragment in fused-cascade mode)
        t0 = time.perf_counter()
        frag.reset()
        kev[s][0].record(stream)
        frag.push(dchunk)
        kev[s][1].record(stream)
        t1 = time.perf_counter()
        result = finish_step()
        t2 = time.perf_counter()
        pm = frag.last_pass_ms()  # events recorded inside push(); the step already synchronised on its result
        if pm is not None:
            pass_ms = [a + b for a, b in zip(pass_ms, pm)]
        if trace is not None:
            trace.append((t1 - t0, t2 - t1, time.perf_counter() - t2))
    ev1.record(stream)
    if trace:
        k = len(trace)
        sys.stderr.write(f"[trace rank {rank}] enqueue reset+push {sum(t[0] for t in trace) / k * 1e3:.3f} ms, finish_step "
                         f"{sum(t[1] for t in trace) / k * 1e3:.3f} ms, last_pass_ms {sum(t[2] for t in trace) / k * 1e3:.3f} ms\n")
    barrier()
    sampler.mark_end()
    launches = ctx.launches - launches0
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = ev0.elapsed_time(ev1)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps
    if world > 1:
        t = torch.tensor([elapsed_ms, kernel_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, kernel_ms = float(t[0]), float(t[1])
    ms_per_step = elapsed_ms / args.steps
    value = n * world / (ms_per_step / 1000.0)
    rows_passed = frag.rows_passed
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, result, {ssb.D_YEAR: "d_year", ssb.C_NATION: "c_nation",
                                                 ssb.OUT_SUM_REVENUE: "sum_lo_revenue", ssb.OUT_SUM_SUPPLYCOST: "sum_lo_supplycost"})

    # ---- e2e: host (pinned) column buffers through the same C-ABI call, H2D inside the timed region ----
    e2e = None
    host_cols = None
    if not args.no_e2e:
        try:
            host_cols = {nm: torch.empty(n, dtype=torch.int32, pin_memory=True) for nm in ssb.Q41_FACT_COLS}
            for nm in ssb.Q41_FACT_COLS:
                host_cols[nm].copy_(cols[nm])
            torch.cuda.synchronize()
        except Exception as ex:  # not enough host memory for the full shard: say so, do not fake it
            host_cols = None
            e2e = {"value": None, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "error": f"pinned host allocation failed: {ex}"}
    def run_e2e(mem):
        morsel = max(1, args.e2e_morsel_rows)

        def e2e_step():
            """one pass over the HOST columns in morsels (what a scan hands over), merge, result to the host"""
            frag.reset()
            for lo in range(0, n, morsel):
                hi = min(n, lo + morsel)
                frag.push(abi.Chunk([(ssb.LO_SLOTS[nm], host_cols[nm][lo:hi].data_ptr(), None, abi.TYPE_INT) for nm in ssb.Q41_FACT_COLS],
                                    num_rows=hi - lo, mem=mem))
            return finish_step()
        r0 = e2e_step()  # warm-up (allocates the staging buffers)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.e2e_steps):
            r0 = e2e_step()
        e1.record(stream)
        barrier()
        ems = e0.elapsed_time(e1) / args.e2e_steps
        if world > 1:
            t = torch.tensor([ems], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t[0])
        d2h = sum(len(c[2]) * abi.TYPE_WIDTH[c[1]] for c in (r0 or result)) if (r0 or result) else 0
        if rank == 0 and r0 is not None and result is not None:
            from starrocks_b200.rows import gpu_rows
            assert gpu_rows(r0) == gpu_rows(result), "e2e (host buffers) result differs from the HBM-resident result"
        return {"value": n * world / (ems / 1000.0), "unit": "rows/s", "d2h_bytes_per_step": d2h, "ms_per_step": ems,
                "steps": args.e2e_steps, "morsel_rows": morsel}

    if host_cols is not None:
        # (1) the columns are read IN PLACE from pinned host memory (SR_MEM_HOST_PINNED): the streaming pass pulls its
        #     key columns over PCIe, the later passes only the 32-byte sectors that hold surviving rows
        e2e = run_e2e(abi.MEM_HOST_PINNED)
        e2e["input_bytes_per_step"] = n * ALGO_BYTES_PER_ROW * world
        e2e["h2d_bytes_per_step"] = int(pcie_bytes_in_place(n, frag.plan()) * world)
        e2e["transfer"] = ("in-place reads of the pinned host columns by the fragment kernels (no staging copy); "
                           "h2d_bytes_per_step = 64-byte bus-block model from the measured pass rates")
        # (2) the same call with a full H2D staging copy of every column (SR_MEM_HOST), for comparison
        full = run_e2e(abi.MEM_HOST)
        full["h2d_bytes_per_step"] = n * ALGO_BYTES_PER_ROW * world
        e2e["staged_copy"] = full
        # (3) the C++ OPERATOR path: DOP pipeline drivers on host threads pull 4096-row chunks and push them into
        #     GpuFragmentSinkOperators sharing one fragment (page-locked double-buffered batches, no blocking call)
        op_bin = os.path.join(ROOT, "starrocks_b200", "host", "bench", "operator_e2e_bench")
        if rank == 0 and world == 1 and not args.no_operator_e2e and os.path.exists(op_bin):
            eff, _ = host_cores()
            dop = max(1, min(8, eff))
            try:
                # frees nothing of ours: the binary creates its own context next to this process's (HBM has room for both)
                r = subprocess.run([op_bin, str(n), str(dop)], capture_output=True, text=True, timeout=600)
                line = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else None
                e2e["operator_api"] = ({"value": line["rows_per_s"], "unit": "rows/s", "seconds": line["seconds"], "dop": line["dop"],
                                        "matches_row_at_a_time_evaluation": line["matches_row_at_a_time_evaluation"],
                                        "fragment_batches": line["fragment_batches"], "h2d_bytes_offered": line["h2d_bytes_offered"],
                                        "d2h_bytes": line["d2h_bytes"], "append_chunk_cpu_seconds_all_threads": line["append_chunk_cpu_seconds_all_threads"],
                                        "need_input_false_polls": line["need_input_false_polls"], "path": line["path"],
                                        "note": "own synthetic SSB-shaped data (same distributions), generated outside the timed region; the timed region holds "
                                                "the 4096-row chunk materialisation of the source, the copies into pinned batches, PCIe and the result D2H"}
                                       if line else {"value": None, "error": (r.stderr or r.stdout)[-300:]})
            except Exception as ex:  # noqa: BLE001
                e2e["operator_api"] = {"value": None, "error": str(ex)}

    # ---- CPU baseline + parity on rank 0 (N = 1 only): the oracle on a bounded sample of the same rows ----
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle
        from starrocks_b200.rows import gpu_rows, oracle_rows
        oracle.lib()
        cores, cores_info = host_cores()
        ojoins, okeep = ssb.build_dims(oracle, dims, ssb.dim_plans_q41())
        if host_cols is not None:
            hnp = {nm: host_cols[nm].numpy() for nm in ssb.Q41_FACT_COLS}
            avail = n
        else:
            avail = min(n, 60_000_000)
            hnp = {nm: cols[nm][:avail].cpu().numpy() for nm in ssb.Q41_FACT_COLS}
        probe = min(avail, 8_000_000)
        dt, _, _ = oracle_run(oracle, ssb, abi, ojoins, hnp, probe, cores)
        sample = args.cpu_sample_rows or int(min(avail, max(probe, (probe / dt) * 15.0)))
        sample = min(sample, avail)
        dt, ores, opassed = oracle_run(oracle, ssb, abi, ojoins, hnp, sample, cores)
        cpu = {"value": sample / dt, "unit": "rows/s", "cores": cores, "kind": "port", "cores_detail": cores_info,
               "sample": f"first {sample} of the same {n} lineorder rows, {cores} pipeline drivers x 4096-row chunks, {dt:.2f} s"}
        # parity at bench size: the GPU path over exactly the sampled rows must equal the oracle bit for bit
        frag.reset()
        sub = abi.Chunk([(ssb.LO_SLOTS[nm], cols[nm][:sample], None, abi.TYPE_INT) for nm in ssb.Q41_FACT_COLS], mem=abi.MEM_DEVICE)
        frag.push(sub)
        got = gpu_rows(frag.agg.result())
        ok = got == oracle_rows(ores) and frag.rows_passed == opassed
        parity = {"rows": sample, "bit_exact": bool(ok), "groups": len(got), "rows_passed": opassed}
        if not ok:
            raise SystemExit("bench.py: GPU result differs from the oracle on the sampled rows -- refusing to report a number")

    # second roofline denominator (SURVEY 8d): read-only 128-bit-load bandwidth over two fact columns (4.8 GB >> L2), best of 5
    read_peak = None
    if rank == 0:
        try:
            import ctypes as _C
            buf = cols["lo_custkey"]
            nbytes = (buf.numel() * 4) // 16 * 16
            best = None
            for _ in range(5):
                r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                r0.record(stream)
                gpu.lib().sr_bandwidth_probe(ctx.h, buf.data_ptr(), nbytes, None)
                gpu.lib().sr_bandwidth_probe(ctx.h, cols["lo_suppkey"].data_ptr(), nbytes, None)
                r1.record(stream)
                torch.cuda.synchronize()
                ms = r0.elapsed_time(r1)
                best = ms if best is None else min(best, ms)
            read_peak = 2 * nbytes / (best / 1000.0) / 1e9
        except Exception as ex:  # noqa: BLE001
            read_peak = None
            sys.stderr.write(f"[bench] read-only bandwidth probe failed: {ex}\n")

    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = n * ALGO_BYTES_PER_ROW / (kernel_ms / 1000.0) / 1e9
        traffic = known_traffic() or {}
        plan = frag.plan()
        kernels = None
        if sum(pass_ms) > 0:
            # per-kernel view: the streaming pass reads its key columns in full (4 B/row each); the gather passes touch
            # single 32-byte sectors, their DRAM traffic is what ncu measured (profiles/traffic.json)
            names = ["k_frag_stream_tests", "k_frag_gather_join", "k_frag_gather_agg"]
            ktr = traffic.get("kernels", {})
            kernels = []
            for nm, ms in zip(names, pass_ms):
                ms /= args.steps
                ent = {"name": nm, "ms": ms, "dram_bytes_per_launch": ktr.get(nm)}
                if nm == "k_frag_stream_tests":
                    ab = n * 4 * max(1, plan["num_stream_joins"])
                    ent.update({"algorithmic_bytes": ab, "achieved_gbs": ab / (ms / 1000.0) / 1e9 if ms > 0 else None,
                                "frac": ab / (ms / 1000.0) / 1e9 / peak if ms > 0 else None,
                                "frac_of_read_only_peak": ab / (ms / 1000.0) / 1e9 / read_peak if (ms > 0 and read_peak) else None})
                kernels.append(ent)
        line = {
            "metric": "rows/sec for SSB Q4.1 hash-join+agg", "value": value, "unit": "rows/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "int32 keys / int64 sums", "data": "synthetic",
            "config": {"workload": f"SSB SF{sf:g} Q4.1 4-way hash join + group-by (scan->probe x4->aggregate), fused fragment",
                       "fact_rows_per_gpu": n, "global_fact_rows": n * world, "dims": {k: int(v) for k, v in sz.items() if k != "lineorder"},
                       "parallelism": f"dp{world}: fact sharded, dimensions replicated (broadcast join), partial aggregates gathered over NCCL",
                       "l2": "inputs (14.4 GB/GPU) >> 126 MB L2, no flush needed", "late_materialization": True,
                       "fragment_plan": plan,
                       "rows_reaching_aggregate_per_gpu": int(rows_passed), "build_ms": build_ms},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic.get("dram_bytes_per_launch"),
                         "kernel": "fragment push = k_frag_stream_tests + k_frag_gather_join + k_frag_gather_agg" if kernels else "k_fragment",
                         "kernel_ms": kernel_ms, "kernels": kernels,
                         "algorithmic_bytes_per_launch": n * ALGO_BYTES_PER_ROW, "peak_source": peak_src,
                         "peak_read_only": read_peak, "peak_read_only_source": "measured in this run: sr_bandwidth_probe (ld.global.nc.v4, xor-reduced) over two 2.4 GB fact columns, best of 5",
                         "note": "achieved = 24 B/row (SURVEY 8d) x rows / CUDA-event duration of one fragment push (all its kernels); "
                                 "late materialisation skips DRAM sectors of later columns whose rows were all filtered out, so the DRAM "
                                 "traffic (ncu) is below the algorithmic bytes and frac may exceed 1"},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "parity": parity,
        }
        print(json.dumps(line))
    frag.close()
    if world > 1:
        dist.destroy_process_group()


def step_tail(frag, final, ctx, gpu, abi, ssb, torch, dist, dev, world, rank, MAXG):
    """N > 1 tail of a step: pull partial states on the device, gather to rank 0 over NCCL (the UNPARTITIONED exchange of
    the two-phase aggregate), final merge by a GPU aggregate on rank 0."""
    from starrocks_b200.distributed import all_gather_partial_states, device_view
    out = frag.agg.pull(mem=abi.MEM_DEVICE)
    g = out.num_rows
    # the pulled columns stay owned by the aggregate handle until its next pull: alias them, no copy
    cols = [device_view(out.cols[k].data, g, abi.TYPE_WIDTH[out.cols[k].type], dev) for k in range(4)]
    pc = all_gather_partial_states(cols, MAXG, dst=0)   # one NCCL collective, one host sync on rank 0
    if rank != 0:
        return None
    final.reset()
    keep = [pc[0].to(torch.int32), pc[1].to(torch.int32), pc[2], pc[3]]
    final.push(abi.Chunk([(ssb.D_YEAR, keep[0], None, abi.TYPE_INT), (ssb.C_NATION, keep[1], None, abi.TYPE_INT),
                          (ssb.OUT_SUM_REVENUE, keep[2], None, abi.TYPE_BIGINT),
                          (ssb.OUT_SUM_SUPPLYCOST, keep[3], None, abi.TYPE_BIGINT)], mem=abi.MEM_DEVICE))
    return final.result()


# ---------------------------------------------------------------------------------------------------
# workload "groupby": BASELINE.json config 5 -- 1e9 rows, 1e8 distinct int64 keys, SUM + COUNT on one B200
# ---------------------------------------------------------------------------------------------------
GROUPBY_BYTES_PER_ROW = 16   # SURVEY.md 8d: key + value in; + 24 B per group out


def splitmix64(x):
    """torch int64 (wrapping) implementation of splitmix64's output function"""
    x = x + (-7046029254386353131)          # 0x9E3779B97F4A7C15 as signed
    z = x
    z = (z ^ ((z >> 30) & ((1 << 34) - 1))) * (-4658895280553007687)   # 0xBF58476D1CE4E5B9
    z = (z ^ ((z >> 27) & ((1 << 37) - 1))) * (-7723592293110705685)   # 0x94D049BB133111EB
    return z ^ ((z >> 31) & ((1 << 33) - 1))


def gen_groupby(torch, dev, n, nk, rank):
    """key int64 = splitmix64(i) mod nk (+ rank * nk: every GPU owns its own key range, as after a hash exchange),
    value int64 U[0, 1000] (SURVEY.md 8d)"""
    keys = torch.empty(n, dtype=torch.int64, device=dev)
    vals = torch.empty(n, dtype=torch.int64, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(20240921 + rank)
    step = 50_000_000
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        i = torch.arange(lo + rank * n, hi + rank * n, dtype=torch.int64, device=dev)
        keys[lo:hi] = torch.remainder(splitmix64(i) & ((1 << 62) - 1), nk) + rank * nk
        vals[lo:hi] = torch.randint(0, 1001, (hi - lo,), dtype=torch.int64, device=dev, generator=g)
        del i
    return keys, vals


def groupby_desc(abi, nk):
    return abi.make_agg_desc([0], [abi.TYPE_BIGINT], fns=[(abi.AGG_SUM, abi.TYPE_BIGINT, 10, [("col", 1)]), (abi.AGG_COUNT_STAR, 0, 11, None)],
                             expected_groups=nk)


def groupby_oracle(oracle, abi, keys_np, vals_np, nk, threads):
    """the CPU arm of the workload: one pipeline driver per thread pre-aggregates its morsels (4096-row chunks), the final
    aggregate merges the partial tables (orc_fragment_run without joins) -- the reference's two-phase plan on one host"""
    chunk = abi.Chunk([(0, keys_np, None, abi.TYPE_BIGINT), (1, vals_np, None, abi.TYPE_BIGINT)])
    t0 = time.perf_counter()
    res, _ = oracle.fragment_run(abi.ScanDesc(), [], groupby_desc(abi, nk), chunk, num_threads=threads)
    return time.perf_counter() - t0, res


def run_reference_groupby(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    from starrocks_b200 import abi
    from oracle import oracle
    oracle.lib()
    n, nk = args.groupby_rows, args.groupby_keys
    cores, cores_info = host_cores()
    sample = args.cpu_sample_rows or min(n, 50_000_000)
    keys, vals = gen_groupby(torch, torch.device("cpu"), sample, nk, 0)
    kn, vn = keys.numpy(), vals.numpy()
    for _ in range(min(args.warmup, 1)):
        groupby_oracle(oracle, abi, kn, vn, nk, cores)
    times = []
    for _ in range(max(1, min(args.steps, 3))):     # bounded: a step is seconds of CPU work
        dt, res = groupby_oracle(oracle, abi, kn, vn, nk, cores)
        times.append(dt)
    value = sample * len(times) / sum(times)
    line = {"impl": "reference", "metric": "rows/sec for high-cardinality group-by (SUM, COUNT)", "value": value, "unit": "rows/s",
            "n_gpus": args.gpus, "steps": len(times), "warmup": min(args.warmup, 1), "ms_per_step": 1000.0 * sum(times) / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": f"group-by {n} rows, {nk} distinct int64 keys, SUM + COUNT", "rows_per_gpu": n, "distinct_keys_per_gpu": nk,
                       "cpu_sample_rows_per_step": sample, "chunk_size": 4096,
                       "note": "StarRocks-semantics CPU restatement (oracle/), NOT the StarRocks BE binary: the BE cannot be built in this image"},
            "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores, "kind": "port", "cores_detail": cores_info,
                             "sample": f"first {sample} of the {n} rows per step, {cores} pipeline drivers pre-aggregating 4096-row chunks + final merge"},
            "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


def run_gpu_groupby(args):
    import torch
    import torch.distributed as dist
    from starrocks_b200 import abi, gpu
    from starrocks_b200.distributed import device_view

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n, nk = args.groupby_rows, args.groupby_keys
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = gpu.Context(local, stream=stream.cuda_stream)
    keys, vals = gen_groupby(torch, dev, n, nk, rank)
    total_v = int(vals.sum().item())
    torch.cuda.synchronize()
    agg = gpu.Agg(ctx, groupby_desc(abi, nk))
    dchunk = abi.Chunk([(0, keys, None, abi.TYPE_BIGINT), (1, vals, None, abi.TYPE_BIGINT)], mem=abi.MEM_DEVICE)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(chunk, out_mem):
        """one pass: push the batch, finish, materialise the result (key, SUM, COUNT per group) in out_mem"""
        agg.reset()
        agg.push(chunk)
        agg.finish()
        return agg.pull(mem=out_mem)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 1)):
        out = step(dchunk, abi.MEM_DEVICE)
    barrier()
    launches0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    sampler.mark_begin()
    ev0.record(stream)
    for s in range(args.steps):
        agg.reset()
        kev[s][0].record(stream)
        agg.push(dchunk)
        kev[s][1].record(stream)
        agg.finish()
        out = agg.pull(mem=abi.MEM_DEVICE)
    ev1.record(stream)
    barrier()
    sampler.mark_end()
    launches = ctx.launches - launches0
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = ev0.elapsed_time(ev1)
    push_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps
    if world > 1:
        t = torch.tensor([elapsed_ms, push_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, push_ms = float(t[0]), float(t[1])
    ms_per_step = elapsed_ms / args.steps
    groups = int(out.num_rows)
    # size-independent checks over the full result (the oracle needs minutes at this size)
    gk = device_view(out.cols[0].data, groups, 8, dev)
    gs = device_view(out.cols[1].data, groups, 8, dev)
    gc = device_view(out.cols[2].data, groups, 8, dev)
    checks = {"count_sum_equals_rows": int(gc.sum().item()) == n, "sum_sum_equals_total": int(gs.sum().item()) == total_v,
              "group_keys_unique": int(torch.unique(gk).numel()) == groups}
    present = torch.zeros(nk, dtype=torch.bool, device=dev)
    for lo in range(0, n, 50_000_000):
        present[keys[lo:min(n, lo + 50_000_000)] - rank * nk] = True
    checks["groups_equal_distinct_keys"] = int(present.sum().item()) == groups
    del present, gk, gs, gc
    if not all(checks.values()):
        raise SystemExit(f"bench.py: group-by invariants violated: {checks}")

    # ---- e2e: host (pinned) key / value columns through sr_agg_push, result pulled to host memory ----
    e2e = None
    if not args.no_e2e:
        try:
            hk = torch.empty(n, dtype=torch.int64, pin_memory=True)
            hv = torch.empty(n, dtype=torch.int64, pin_memory=True)
            hk.copy_(keys)
            hv.copy_(vals)
            torch.cuda.synchronize()
            hchunk = abi.Chunk([(0, hk.data_ptr(), None, abi.TYPE_BIGINT), (1, hv.data_ptr(), None, abi.TYPE_BIGINT)], num_rows=n, mem=abi.MEM_HOST)
            step(hchunk, abi.MEM_HOST)   # warm-up: allocates the staging + pinned result buffers
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.e2e_steps):
                ho = step(hchunk, abi.MEM_HOST)
            e1.record(stream)
            barrier()
            ems = e0.elapsed_time(e1) / args.e2e_steps
            if world > 1:
                t = torch.tensor([ems], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ems = float(t[0])
            assert ho.num_rows == groups
            e2e = {"value": n * world / (ems / 1000.0), "unit": "rows/s", "ms_per_step": ems, "steps": args.e2e_steps,
                   "h2d_bytes_per_step": n * GROUPBY_BYTES_PER_ROW * world, "d2h_bytes_per_step": groups * 24 * world,
                   "transfer": "sr_agg_push on pinned host columns (staged H2D copy on the context's stream), sr_agg_pull into pinned host buffers"}
            del hk, hv
        except Exception as ex:  # noqa: BLE001 -- not enough pinned host memory: say so, do not fake it
            e2e = {"value": None, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": str(ex)}

    # ---- CPU baseline + parity (rank 0, N = 1): the oracle on the first rows of the same data ----
    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle
        oracle.lib()
        cores, cores_info = host_cores()
        sample = args.cpu_sample_rows or min(n, 50_000_000)
        kn, vn = keys[:sample].cpu().numpy(), vals[:sample].cpu().numpy()
        dt, ores = groupby_oracle(oracle, abi, kn, vn, nk, cores)
        cpu = {"value": sample / dt, "unit": "rows/s", "cores": cores, "kind": "port", "cores_detail": cores_info,
               "sample": f"first {sample} of the same {n} rows, {cores} pipeline drivers pre-aggregating 4096-row chunks + final merge, {dt:.2f} s"}
        oo = ores.output()
        order = np.argsort(oo[0][1], kind="stable")
        agg.reset()
        agg.push(abi.Chunk([(0, keys[:sample], None, abi.TYPE_BIGINT), (1, vals[:sample], None, abi.TYPE_BIGINT)], mem=abi.MEM_DEVICE))
        agg.finish()
        po = agg.pull(mem=abi.MEM_DEVICE)
        pg = int(po.num_rows)
        pk = device_view(po.cols[0].data, pg, 8, dev)
        srt = torch.argsort(pk)
        ok = pg == len(order)
        for c in range(3):
            if not ok:
                break
            got = device_view(po.cols[c].data, pg, 8, dev)[srt].cpu().numpy()
            ok = bool(np.array_equal(got, oo[c][1][order]))
        parity = {"rows": sample, "bit_exact": bool(ok), "groups": pg}
        if not ok:
            raise SystemExit("bench.py: GPU group-by differs from the oracle on the sampled rows -- refusing to report a number")

    if rank == 0:
        peak, peak_src = measured_peak()
        abytes = n * GROUPBY_BYTES_PER_ROW + groups * 24
        achieved = abytes / (ms_per_step / 1000.0) / 1e9
        traffic = (known_traffic() or {}).get("groupby_dram_bytes_per_launch")
        line = {
            "metric": "rows/sec for high-cardinality group-by (SUM, COUNT)", "value": n * world / (ms_per_step / 1000.0), "unit": "rows/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": f"group-by {n} rows, {nk} distinct int64 keys, SUM + COUNT", "rows_per_gpu": n, "distinct_keys_per_gpu": nk,
                       "groups_per_gpu": groups, "parallelism": f"dp{world}: one key range per GPU (rows already hash-exchanged), no collective",
                       "l2": "inputs (16 GB/GPU) >> 126 MB L2, no flush needed"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "kernel": "sr_agg_push (k_aggp_scatter x 2 + k_aggp_apply) + result materialisation (k_agg_count / k_agg_emit)",
                         "kernel_ms": ms_per_step, "push_ms": push_ms, "algorithmic_bytes_per_launch": abytes, "peak_source": peak_src,
                         "note": "achieved = (16 B/row in + 24 B/group out, SURVEY 8d) / CUDA-event duration of one step (reset, push, finish, emit); "
                                 "the partitioned push moves every row through HBM two more times (two scatter levels)"},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "parity": parity, "checks": checks,
        }
        print(json.dumps(line))
    agg.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.workload == "q3":
        if a.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the CPU arm of the Q3 workload is the oracle check inside tools/q3_distributed.py (--check oracle)"}))
        else:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import q3_distributed
            q3_distributed.main(q3_distributed.parse(["--sf", str(a.sf if a.sf != 100.0 else 300.0), "--steps", str(a.steps), "--warmup", str(a.warmup)]))
    elif a.workload == "q95":
        if a.impl == "reference":
            if int(os.environ.get("RANK", "0")) == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the CPU arm of the Q95 workload is the oracle check inside tools/q95_distributed.py (--check oracle)"}))
        else:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import q95_distributed
            world = int(os.environ.get("WORLD_SIZE", "1"))
            q95_distributed.main(q95_distributed.parse(["--sf", str(a.sf if a.sf != 100.0 else 125.0 * world), "--steps", str(a.steps), "--warmup", str(a.warmup)]))
    elif a.workload == "groupby":
        run_reference_groupby(a) if a.impl == "reference" else run_gpu_groupby(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_gpu(a)
