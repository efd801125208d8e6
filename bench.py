#!/usr/bin/env python
"""bench.py — groupby-agg rows/sec on B200 (BASELINE.json metric), roofline and CPU baseline.

Workload (config.workload): BASELINE.json configs[1] "2B-row int64 2-col, 1M-group groupby SUM/COUNT on
1xB200"; with --gpus N > 1 it is configs[3] (the same 2B rows sharded across N GPUs, strong scaling, one
hash-partition exchange of the partial aggregates over NCCL).  One step = one whole operator lifetime over
the batch: init state -> consume all local rows -> (exchange) -> finalize -> produce.

  value     rows/s with the input columns already resident in HBM (CUDA events, max over ranks)
  e2e       rows/s through the same public API with HOST (pinned) input columns and a host copy of the result
  roofline  consume kernel: 16 B/row (8 B key + 8 B value, SURVEY.md §8d) / its mean launch time, measured with
            CUDA events on the kernel's stream, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle (reference algorithm shape, one rank per host thread) on a bounded sample

`--impl reference` times only that CPU restatement (the reference runtime cannot be built here: no MPI).

The line also carries `config.no_hint` (the same steps without the expected_groups hint, which the reference's API does not
have; `--no-hint` makes that the headline run).  `--dump-outputs DIR` writes the result of the last timed step (float64
DIR/<column>.npy, rows ordered by key) so that two builds can be compared array for array on the same seeded input.
Other workloads, each printing the same kind of line:
  --workload join                           BASELINE.json configs[2], benchmarks/join_bench.py
  --workload shuffle                        raw-row variant of configs[3], benchmarks/shuffle_bench.py
  --aggs F1,F2.. [--nullable] [--key-dtype int32] [--val-dtype int32]
                                            other signatures of configs[1], benchmarks/groupby_variant_bench.py
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "groupby-agg rows/sec"
UNIT = "rows/s"
BYTES_PER_ROW = 16  # algorithmic bytes of the hash-aggregate scan (SURVEY.md §8d)
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full captures (profiles/):
# filled in from profiles/r01_*.txt for the 2^26-row launch of the default workload; None = not captured
# spg: profiles/r01_spg_ncu_summary.txt, K1 1.074+1.019 GB + K2 1.123+0.004 GB per 2^26-row launch pair (3x the
# algorithmic 1.074 GB by design: rows are written to and re-read from owner buckets).
# direct: profiles/r01_direct_ncu_summary.txt (2^27-row launch, bucketized variant): 10.99 + 0.18 GB.
# Both are DRAM bytes per ROW of a launch (measured bytes / rows of the captured launch); one launch of the timed run
# moves that figure x its own row count (launches are 2^27 rows now, the captures above were taken on 2^26 / 2^27).
# spgn (narrow bucket rows, the path the default workload takes since round 2): profiles/r02_launches.txt (105 launches of the
# shipping 2^27-row kernels): K1n 2.133 + 1.029 GB, K2n 1.116 + 0.000 GB = 4.279 GB = 31.9 B/row (16 read + 8 bucket write +
# 8 bucket read by design).
TRAFFIC_PER_ROW = {"spg": 3.220e9 / (1 << 26), "spgn": 4.279e9 / (1 << 27), "direct": 11.17e9 / (1 << 27)}
DUMP_BYTES = 64 << 20  # --dump-outputs writes at most this much in all


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=2_000_000_000, help="total rows over all GPUs")
    ap.add_argument("--groups", type=int, default=1_000_000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-sample-rows", type=int, default=1_000_000_000)
    ap.add_argument("--ref-sample-rows", type=int, default=512_000_000)
    # --workload join: BASELINE.json configs[2] (benchmarks/join_bench.py); the default workload is the contract's configs[1] / [3]
    ap.add_argument("--workload", default="groupby", choices=["groupby", "join", "shuffle"])
    ap.add_argument("--n-dest", type=int, default=8, help="shuffle workload at N=1: destinations to partition into")
    ap.add_argument("--aggs", default="sum,count", help="groupby aggregate functions; anything but sum,count runs the variant bench")
    ap.add_argument("--nullable", action="store_true", help="groupby variant: nullable key (1 %% NA) and value (10 %% NA) columns")
    ap.add_argument("--key-dtype", default="int64", choices=["int64", "int32"])
    ap.add_argument("--val-dtype", default="int64", choices=["int64", "int32"])
    ap.add_argument("--no-hint", action="store_true", help="do not pass the exact cardinality as expected_groups")
    ap.add_argument("--build-rows", type=int, default=100_000_000)
    ap.add_argument("--probe-rows", type=int, default=1_000_000_000)
    ap.add_argument("--probe-batch", type=int, default=250_000_000)
    ap.add_argument("--sample-lo", type=int, default=1000, help="join parity: sorted row-set equality for keys in [lo, hi)")
    ap.add_argument("--sample-hi", type=int, default=1400)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step as float64 DIR/<column>.npy, "
                    "rows ordered by key (default groupby workload, one process)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clock / throttle-reason sampler running during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.p = None
        self.path = f"/tmp/b200_clocks_{os.getpid()}.csv"
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        # wait for the first sample: nvidia-smi's start-up (NVML initialisation over all GPUs of the box, 0.2 - 1 s) takes driver
        # locks that stall CUDA calls of the benchmark process; it has to be over before the timed region starts (an 8-GPU run
        # whose 30 ms timed region overlapped it lost 1.4 ms per step)
        t0 = time.time()
        while self.p is not None and time.time() - t0 < 5.0:
            try:
                if os.path.getsize(self.path) > 0:
                    break
            except OSError:
                pass
            if self.p.poll() is not None:
                break
            time.sleep(0.02)

    def stop(self):
        if self.p is None:
            return None
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for ln in open(self.path):
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def pick_threads(keys_np, vals_np) -> int:
    """The oracle's one-rank-per-thread SPMD shape does not scale linearly on big hosts (random access, shared LLC):
    try a few rank counts on a small prefix and keep the fastest (reported as `cores`)."""
    from oracle import oracle as O

    avail = host_threads()
    cands = sorted({t for t in (avail, avail // 2, avail // 4, 32, 16) if 1 <= t <= avail})
    n = min(len(keys_np), 32_000_000)
    best, best_rate = avail, 0.0
    for t in cands:
        t0 = time.perf_counter()
        O.groupby_sum_count_mt(keys_np[:n], vals_np[:n], t)
        rate = n / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = t, rate
    return best


def run_cpu_baseline(keys_np, vals_np, threads: int):
    """Times the oracle's SPMD restatement; returns (rows/s, seconds, n_groups, checksums)."""
    from oracle import oracle as O

    t0 = time.perf_counter()
    ng, cs = O.groupby_sum_count_mt(keys_np, vals_np, threads)
    dt = time.perf_counter() - t0
    return len(keys_np) / dt, dt, ng, cs


def reference_arm(args):
    """bench.py --impl reference: the reference's CPU algorithm (oracle port; the MPI runtime is unbuildable here,
    DESIGN.md) on all host threads, each step one bounded sample of the same synthetic workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O

    n = min(args.ref_sample_rows, args.rows)
    keys, vals = O.synth_fill(0, n, args.groups, args.seed)
    threads = pick_threads(keys, vals)
    for _ in range(max(args.warmup, 0)):
        run_cpu_baseline(keys, vals, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, _, ng, cs = run_cpu_baseline(keys, vals, threads)
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    sample = f"first {n} rows of the {args.rows}-row table per step, {args.groups} groups"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": workload_name(args), "rows": args.rows, "groups": args.groups, "aggs": ["sum", "count"],
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def write_outputs(out_dir, cols):
    """--dump-outputs: the columns {name: device tensor} a caller of the timed path received, as DIR/<name>.npy in float64.
    Rows are ordered by the first (key) column: the library's row order is not part of its result.  Above DUMP_BYTES in all,
    a fixed seeded sample of the ordered rows is written, the same rows for the same arguments, so that the files of two builds
    can be compared array for array."""
    import numpy as np
    import torch

    names = list(cols)
    order = torch.argsort(cols[names[0]])
    cap = DUMP_BYTES // (8 * len(names))
    if order.numel() > cap:
        pick = np.sort(np.random.default_rng(0).choice(order.numel(), cap, replace=False))
        order = order[torch.from_numpy(pick).to(order.device)]
    os.makedirs(out_dir, exist_ok=True)
    for name in names:
        np.save(os.path.join(out_dir, f"{name}.npy"), cols[name][order].cpu().numpy().astype(np.float64))


def workload_name(args):
    if args.gpus == 1:
        return f"{args.rows}-row int64 2-col, {args.groups}-group groupby SUM/COUNT on 1xB200 (BASELINE.json configs[1])"
    return (f"{args.rows}-row {args.groups}-group groupby SUM/COUNT sharded across {args.gpus}xB200, hash-partition "
            f"exchange of partial aggregates over NCCL (BASELINE.json configs[3])")


def main():
    args = parse_args()
    variant = args.aggs.replace(" ", "") != "sum,count" or args.nullable or args.key_dtype != "int64" or args.val_dtype != "int64"
    if args.dump_outputs and (args.workload != "groupby" or args.impl != "b200" or variant):
        sys.exit("--dump-outputs is implemented for the default groupby workload only")
    if args.workload == "join":
        from benchmarks import join_bench

        join_bench.run(args, ClockSampler, peaks)
        return
    if args.workload == "shuffle":
        from benchmarks import shuffle_bench

        shuffle_bench.run(args, ClockSampler, peaks)
        return
    if args.impl == "reference":
        reference_arm(args)
        return
    if variant:
        from benchmarks import groupby_variant_bench

        groupby_variant_bench.run(args, ClockSampler, peaks)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from bodo_b200 import _lib, synth
    from bodo_b200.streaming import groupby as G
    from bodo_b200.table import Column, Table

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if args.dump_outputs and world > 1:
        sys.exit("--dump-outputs writes the result of one process: run it with --gpus 1")
    _lib.require_gpu()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.current_stream(dev)
    stream_ptr = stream.cuda_stream

    # strong scaling: the 2B-row table is split into contiguous row slices (dist_get_start/end style)
    chunk = (args.rows + world - 1) // world
    row0 = min(rank * chunk, args.rows)
    n_local = min(chunk, args.rows - row0)
    keys = torch.empty(n_local, dtype=torch.int64, device=dev)
    vals = torch.empty(n_local, dtype=torch.int64, device=dev)
    synth.device_fill(keys, vals, row0, args.groups, args.seed, stream_ptr)
    torch.cuda.synchronize(dev)
    expect_sum = int(vals.sum().item())  # wraps like the int64 SUM does
    table = Table([Column(keys), Column(vals)], ["key", "val"])
    exp_groups_local = 0 if args.no_hint else args.groups

    stats = {}

    def one_step(tab, collect=False, profile=False, to_host=False, hint=None, keep=False):
        st = G.init_groupby_state(-1, (0,), ("sum", "count"), (0, 1, 2), (1, 1), parallel=world > 1,
                                  expected_groups=exp_groups_local if hint is None else hint,
                                  output_batch_size=1 << 40, device=local_rank, stream=stream_ptr)
        st._ensure(tab)
        if profile:
            G.get_metric(st, 100)
        G.groupby_build_consume_batch(st, tab, True, True)
        out, last = G.groupby_produce_output_batch(st, True)
        assert last
        res = None
        if to_host:
            res = [c.values_numpy(stream_ptr) for c in out.columns]
            stats["d2h"] = sum(a.nbytes for a in res)
        if keep:  # the output columns are the state's memory: copy them before it is deleted
            stats["kept"] = {nm: torch.as_tensor(c.data, device=dev)[:out.n_rows].clone() for nm, c in zip(out.names, out.columns)}
        if collect:
            cols = [torch.as_tensor(c.data, device=dev) for c in out.columns]
            stats["n_out"] = out.n_rows
            stats["sum_of_sums"] = int(cols[1].sum().item()) if out.n_rows else 0
            stats["sum_of_counts"] = int(cols[2].sum().item()) if out.n_rows else 0
            stats["per_group"] = per_group_check(cols, out.n_rows)
            stats["launches"] = G.get_metric(st, 4)
            if profile:
                stats["consume_us"] = G.get_metric(st, 6)
                stats["consume_launches"] = G.get_metric(st, 7)
                stats["spg_launches"] = G.get_metric(st, 8)
                stats["spgn_launches"] = G.get_metric(st, 14)
        G.delete_groupby_state(st)
        return res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def per_group_check(cols, n_out):
        """EVERY group this rank produced against an independent recomputation (torch scatter-adds over the raw rows of all
        ranks, dense by key: the synthetic keys are 0 .. groups-1), and its placement: hash_to_rank(key) == rank — the
        reference's ownership rule (bodo/libs/_shuffle.h:5-7).  Returns (ok, n_bad, n_misplaced, n_groups_expected_total)."""
        ref_sum = torch.zeros(args.groups, dtype=torch.int64, device=dev)
        ref_cnt = torch.zeros(args.groups, dtype=torch.int64, device=dev)
        step_rows = 1 << 27
        for r0 in range(0, n_local, step_rows):  # bounded temporaries
            kk = keys[r0:r0 + step_rows]
            ref_sum.index_add_(0, kk, vals[r0:r0 + step_rows])
            ref_cnt += torch.bincount(kk, minlength=args.groups)
        if world > 1:
            dist.all_reduce(ref_sum)
            dist.all_reduce(ref_cnt)
        n_expected = int((ref_cnt > 0).sum().item())
        if n_out == 0:
            return True, 0, 0, n_expected
        okeys = cols[0][:n_out]
        in_range = (okeys >= 0) & (okeys < args.groups)
        safe = torch.where(in_range, okeys, torch.zeros_like(okeys))
        bad = (~in_range) | (cols[1][:n_out] != ref_sum[safe]) | (cols[2][:n_out] != ref_cnt[safe])
        dup = okeys.numel() - torch.unique(okeys).numel()
        n_misplaced = 0
        if world > 1:
            dest = torch.empty(n_out, dtype=torch.int32, device=dev)
            from bodo_b200.table import CTable
            ct = CTable(Table([Column(okeys.contiguous())], ["key"]))
            _lib.check(_lib.lib().b200_hash_to_rank(ct.ptr, world, _lib.ffi.cast("int32_t*", dest.data_ptr()), _lib.ffi.cast("void*", stream_ptr)),
                       "hash_to_rank")
            torch.cuda.synchronize(dev)
            n_misplaced = int((dest != rank).sum().item())
        n_bad = int(bad.sum().item()) + dup
        return (n_bad == 0 and n_misplaced == 0), n_bad, n_misplaced, n_expected

    # the clock sampler starts before the warm-up (nvidia-smi needs ~0.2 s to deliver its first sample and a short timed region
    # would otherwise end before it): warm-up and timed steps are the same workload, every sample is taken under load
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()  # rank 0 may have waited for nvidia-smi: line the ranks up again before the first collective step
    for _ in range(max(args.warmup, 0)):
        one_step(table)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for i in range(args.steps):
        one_step(table, keep=bool(args.dump_outputs) and i == args.steps - 1)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        write_outputs(args.dump_outputs, stats.pop("kept"))

    # the same steps WITHOUT the expected_groups hint (the reference's API has no such argument: a drop-in caller gets this
    # route — the state learns the cardinality from a 2^20-row prefix through the direct kernel, then takes the same kernels)
    barrier()
    nh0, nh1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    one_step(table, hint=0)
    barrier()
    nh0.record(stream)
    for _ in range(args.steps):
        one_step(table, hint=0)
    nh1.record(stream)
    barrier()
    nh = torch.tensor([nh0.elapsed_time(nh1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(nh, op=dist.ReduceOp.MAX)
    no_hint_ms = float(nh[0].item())

    # untimed: one profiled step (per-launch CUDA events inside the library) + result check
    one_step(table, collect=True, profile=True)
    barrier()
    pg_ok, pg_bad, pg_misplaced, pg_expected = stats["per_group"]
    tot = torch.tensor([ms, float(stats["n_out"]), float(pg_bad + pg_misplaced)], dtype=torch.float64, device=dev)
    chk = torch.tensor([stats["sum_of_sums"], stats["sum_of_counts"], expect_sum], dtype=torch.int64, device=dev)
    if world > 1:
        mx = tot.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dist.all_reduce(chk, op=dist.ReduceOp.SUM)
        ms = float(mx[0].item())
    n_groups_total = int(tot[1].item())
    per_group_ok = int(tot[2].item()) == 0 and n_groups_total == pg_expected
    check_ok = int(chk[1].item()) == args.rows and int(chk[0].item()) == int(chk[2].item()) and per_group_ok

    value = args.rows * args.steps / (ms * 1e-3)
    peak, peak_kind = peaks()
    kern_us = stats.get("consume_us", 0)
    n_launch = max(stats.get("consume_launches", 1), 1)
    achieved = (BYTES_PER_ROW * n_local / 1e9) / (kern_us * 1e-6) if kern_us else None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": TRAFFIC_PER_ROW["spgn" if stats.get("spgn_launches") else "spg" if stats.get("spg_launches") else "direct"] * n_local / n_launch,
                "peak_kind": peak_kind,
                "kernel": ("spgn_partition_kernel<true,true> + spgn_aggregate_kernel<true,true> (narrow bucket rows; one launch = the pair)"
                           if stats.get("spgn_launches") else
                           "spg_partition_tma_kernel<true,true> + spg_aggregate_kernel<true,true> (one launch = the pair)"
                           if stats.get("spg_launches") else "groupby_consume_i64_sumcount_kernel<true,true>"),
                "launches_per_step": n_launch, "avg_launch_ms": kern_us / 1e3 / n_launch,
                "algorithmic_bytes_per_launch": BYTES_PER_ROW * n_local / n_launch}

    # ---- e2e: same API, HOST (pinned) input columns, result copied back to the host every step ----
    e2e = None
    if not args.no_e2e:
        try:
            hk = torch.empty(n_local, dtype=torch.int64, pin_memory=True)
            hv = torch.empty(n_local, dtype=torch.int64, pin_memory=True)
            hk.copy_(keys); hv.copy_(vals)
            torch.cuda.synchronize(dev)
            htab = Table([Column(hk.numpy()), Column(hv.numpy())], ["key", "val"])
            one_step(htab, to_host=True)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record(stream)
            for _ in range(args.e2e_steps):
                one_step(htab, to_host=True)
            e1.record(stream)
            barrier()
            wall = time.perf_counter() - t0
            ems = max(e0.elapsed_time(e1), wall * 1e3 * 0.0)  # device span; host wall reported beside it
            emax = torch.tensor([ems, wall * 1e3], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(emax, op=dist.ReduceOp.MAX)
            ems, wall_ms = float(emax[0].item()), float(emax[1].item())
            e2e = {"value": args.rows * args.e2e_steps / (max(ems, wall_ms) * 1e-3), "unit": UNIT,
                   "h2d_bytes_per_step": 16 * n_local, "d2h_bytes_per_step": int(stats.get("d2h", 0)),
                   "steps": args.e2e_steps, "ms_per_step": max(ems, wall_ms) / args.e2e_steps, "host_memory": "pinned"}
            del hk, hv, htab
        except Exception as ex:  # e.g. not enough pinnable host memory
            e2e = {"value": None, "unit": UNIT, "error": str(ex)[:200]}

    # ---- CPU baseline on rank 0 at N == 1 ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ns = min(args.cpu_sample_rows, n_local)
        while cpu is None and ns >= 1_000_000:
            try:
                kn = keys[:ns].cpu().numpy()
                vn = vals[:ns].cpu().numpy()
                threads = pick_threads(kn, vn)
                rps, secs, ng, cs = run_cpu_baseline(kn, vn, threads)
                cpu = {"value": rps, "unit": UNIT, "cores": threads, "kind": "port", "seconds": secs,
                       "sample": f"first {ns} rows of the {args.rows}-row table, {ng} groups (oracle SPMD restatement, one rank per thread)"}
            except MemoryError:  # host smaller than expected: halve the sample
                ns //= 2

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": {"workload": workload_name(args), "rows": args.rows, "groups": args.groups, "aggs": ["sum", "count"],
                       "rows_per_gpu": n_local, "l2": "inputs (16 B/row x rows_per_gpu) exceed the 126 MB L2; no flush needed",
                       "step": "init state + consume + exchange + finalize + produce", "result_groups": n_groups_total,
                       "expected_groups_hint": exp_groups_local,
                       "no_hint": {"value": args.rows * args.steps / (no_hint_ms * 1e-3), "ms_per_step": no_hint_ms / args.steps,
                                   "note": "same steps with expected_groups=0 (what a caller of the reference's API passes)"},
                       "result_check": ("per-group ok: every group's SUM and COUNT equal an independent device recomputation over all ranks' rows"
                                        + ("; every group sits on hash_to_rank(key)" if world > 1 else "")) if check_ok else "MISMATCH"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(stats.get("launches", 0)) * args.steps,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if not check_ok:
        sys.exit(3)


if __name__ == "__main__":
    main()
