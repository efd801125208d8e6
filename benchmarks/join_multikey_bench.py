"""Multi-column equi-join keys: BASELINE.json configs[2] (hash inner join, 100 M build x 1 B probe rows, 2 payload columns per
side, 250 M-row probe batches, 1 x B200) with the int64 key split into two key columns, against the single-key join on the
combined key over the same rows.

    python benchmarks/join_multikey_bench.py [--steps K] [--warmup W]

  keys      k1 = key >> 10 (int64), k2 = key & 1023 (int32); build keys are a permutation of [0, build_rows), so build tuples
            are unique and every probe row has exactly one match.  The tuple join takes the fused multi-key probe
            (join_probe_fast_mk_kernel<2>: a Slot16 table of tuple tags + packed build rows); the single-key arm takes the
            inline-payload Slot32 probe (join_probe_inline_kernel), the kernel bench.py --workload join measures.
  step      one whole operator lifetime, as in benchmarks/join_bench.py: init state -> build (one batch) -> probe batches, every
            batch materialising its joined rows (tuple arm: k1, k2, b1, b2, p1, p2; single-key arm: k, b1, b2, p1, p2).
            The two arms alternate step by step in one process; each step is timed with CUDA events on the operator's stream.
  parity    untimed, at full size, tuple arm: output row count; sum mod 2^64 of every output column against an
            inverse-permutation torch recomputation; sorted row-set equality on a sampled key range.  Exit code 3 on a mismatch.

Prints one JSON line in bench.py's shape (value = tuple-arm probe rows/s), with the single-key rate, their ratio, per-launch
probe times of the tuple arm, and the card's name and power limit read in the same run.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "multi-key hash-join probe rows/sec"
UNIT = "rows/s"
MASK64 = (1 << 64) - 1


def parse_args(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--build-rows", type=int, default=100_000_000)
    ap.add_argument("--probe-rows", type=int, default=1_000_000_000)
    ap.add_argument("--probe-batch", type=int, default=250_000_000)
    ap.add_argument("--sample-lo", type=int, default=1000, help="parity: sorted row-set equality for combined keys in [lo, hi)")
    ap.add_argument("--sample-hi", type=int, default=1400)
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def gpu_info() -> dict:
    """Name, power limit and max SM clock of GPU 0 (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"name": out[0].strip(), "power_limit_w": float(out[1]), "sm_max_mhz": float(out[2])}
    except Exception as ex:
        import torch

        return {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "error": str(ex)[:120]}


def u64sum(t) -> int:
    """sum mod 2^64 of an integer / float64 tensor (floats by bit pattern, narrow integers widened)."""
    import torch

    v = t.view(torch.int64) if t.element_size() == 8 else t.to(torch.int64)
    return int(v.sum().item()) & MASK64


def main(argv=None):
    args = parse_args(argv)
    import torch

    from bench import ClockSampler
    from bodo_b200 import _lib, synth
    from bodo_b200.streaming import join as J
    from bodo_b200.table import Column, Table

    _lib.require_gpu()
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    sp = stream.cuda_stream
    nb, npr, batch = args.build_rows, args.probe_rows, args.probe_batch

    # the rows of benchmarks/join_bench.py: build keys a permutation of [0, nb), probe keys uniform in [0, nb)
    bk = torch.randperm(nb, device=dev, dtype=torch.int64, generator=torch.Generator(device=dev).manual_seed(3))
    b1 = torch.empty(nb, dtype=torch.int64, device=dev)
    b2 = torch.empty(nb, dtype=torch.float64, device=dev)
    synth.device_fill(None, b1, 0, 1, 31, sp)
    synth.device_fill(None, b2, 0, 1, 32, sp)
    pk = torch.empty(npr, dtype=torch.int64, device=dev)
    p1 = torch.empty(npr, dtype=torch.int64, device=dev)
    p2 = torch.empty(npr, dtype=torch.float64, device=dev)
    synth.device_fill(pk, p1, 0, nb, 41, sp)
    synth.device_fill(None, p2, 0, 1, 42, sp)
    bk1, bk2 = bk >> 10, (bk & 1023).to(torch.int32)
    pk1, pk2 = pk >> 10, (pk & 1023).to(torch.int32)
    torch.cuda.synchronize(dev)

    arms = {
        "tuple": dict(build=Table([Column(bk1), Column(bk2), Column(b1), Column(b2)], ["k1", "k2", "b1", "b2"]), probe=(pk1, pk2, p1, p2),
                      pnames=["k1", "k2", "p1", "p2"], keys=(0, 1), kept=([0, 1, 2, 3], [2, 3])),
        "single": dict(build=Table([Column(bk), Column(b1), Column(b2)], ["k", "b1", "b2"]), probe=(pk, p1, p2),
                       pnames=["k", "p1", "p2"], keys=(0,), kept=([0, 1, 2], [1, 2])),
    }
    stats = {}

    def one_step(arm, verify=False, profile=False):
        a = arms[arm]
        st = J.init_join_state(-1, a["keys"], a["keys"], tuple(a["build"].names), tuple(a["pnames"]), False, False,
                               expected_build_rows=nb, device=0, stream=sp)
        J.join_build_consume_batch(st, a["build"], True)
        out_rows, sums, sample_rows, evs = 0, None, [], []
        for r0 in range(0, npr, batch):
            r1 = min(npr, r0 + batch)
            t = Table([Column(c[r0:r1]) for c in a["probe"]], list(a["pnames"]))
            if profile:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
            out, _, _ = J.join_probe_consume_batch(st, t, r1 == npr, True, a["kept"])
            if profile:
                e1.record(stream)
                evs.append((e0, e1))
            out_rows += out.n_rows
            if verify:
                cols = [torch.as_tensor(c.data, device=dev)[: out.n_rows] for c in out.columns]
                part = [u64sum(c) for c in cols]
                sums = part if sums is None else [(x + y) & MASK64 for x, y in zip(sums, part)]
                key = (cols[0] << 10) | cols[1].to(torch.int64)
                m = (key >= args.sample_lo) & (key < args.sample_hi)
                sample_rows.append(torch.stack([c.view(torch.int64) if c.element_size() == 8 else c.to(torch.int64) for c in cols], 1)[m].cpu())
        stats[arm] = {"launches": J.get_metric(st, 4), "fused_probes": J.get_metric(st, 5), "inline_probes": J.get_metric(st, 6)}
        J.delete_join_state(st)
        if profile:
            torch.cuda.synchronize(dev)
            stats[arm]["probe_ms"] = [e0.elapsed_time(e1) for e0, e1 in evs]
        return out_rows, sums, sample_rows

    info = gpu_info()
    sampler = ClockSampler(0)
    for _ in range(max(args.warmup, 0)):
        one_step("tuple")
        one_step("single")
    ms = {"tuple": 0.0, "single": 0.0}
    for _ in range(args.steps):  # alternate the arms step by step
        for arm in ("tuple", "single"):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record(stream)
            one_step(arm)
            e1.record(stream)
            torch.cuda.synchronize(dev)
            ms[arm] += e0.elapsed_time(e1)
    clocks = sampler.stop()

    # ---- untimed: profiled tuple step + parity at full size ----
    out_rows, sums, sample_rows = one_step("tuple", verify=True, profile=True)
    inv = torch.empty(nb, dtype=torch.int64, device=dev)
    inv[bk] = torch.arange(nb, dtype=torch.int64, device=dev)
    exp_sums, exp_sample = [0] * 6, []
    for r0 in range(0, npr, batch):
        r1 = min(npr, r0 + batch)
        kk = pk[r0:r1]
        bi = inv[kk]
        cols = [bk1[bi], bk2[bi], b1[bi], b2[bi], p1[r0:r1], p2[r0:r1]]
        exp_sums = [(x + u64sum(c)) & MASK64 for x, c in zip(exp_sums, cols)]
        m = (kk >= args.sample_lo) & (kk < args.sample_hi)
        exp_sample.append(torch.stack([c.view(torch.int64) if c.element_size() == 8 else c.to(torch.int64) for c in cols], 1)[m].cpu())
    del inv
    got_s = torch.cat(sample_rows) if sample_rows else torch.zeros((0, 6), dtype=torch.int64)
    exp_s = torch.cat(exp_sample)

    def sort_rows(t):
        return t[sorted(range(t.shape[0]), key=lambda i: tuple(t[i].tolist()))]

    sample_ok = got_s.shape == exp_s.shape and bool((sort_rows(got_s) == sort_rows(exp_s)).all())
    check_ok = out_rows == npr and sums == exp_sums and sample_ok
    paths_ok = stats["tuple"]["fused_probes"] >= 1 and stats["single"]["inline_probes"] >= 1

    rate = {arm: npr * args.steps / (ms[arm] * 1e-3) for arm in ms}
    pms = stats["tuple"]["probe_ms"]
    print(json.dumps({
        "metric": METRIC, "value": rate["tuple"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms["tuple"] / args.steps, "higher_is_better": True, "scaling": "strong", "dtype": "int64 + int32 keys",
        "data": "synthetic",
        "config": {"workload": f"hash inner join {npr} x {nb} on (k1 int64, k2 int32), 2 payload cols per side on 1xB200 "
                               "(BASELINE.json configs[2] with the key split in two columns)",
                   "build_rows": nb, "probe_rows": npr, "probe_batch": batch, "out_rows": out_rows,
                   "step": "init state + build (tag table, CSR pass, row pack) + probe batches with output materialisation",
                   "result_check": ("ok: row count, sum mod 2^64 of all 6 output columns vs inverse-permutation gathers, sorted row-set "
                                    f"equality for keys in [{args.sample_lo}, {args.sample_hi}) ({got_s.shape[0]} rows)") if check_ok else "MISMATCH",
                   "paths": "ok" if paths_ok else "UNEXPECTED"},
        "kernel": "join_probe_fast_mk_kernel<2> (fused probe, unique build tuples)",
        "probe_launch_ms": pms, "launches_per_step": len(pms), "gpu_launches": int(stats["tuple"]["launches"]) * args.steps,
        "single_key": {"value": rate["single"], "unit": UNIT, "ms_per_step": ms["single"] / args.steps,
                       "kernel": "join_probe_inline_kernel<2,2> (inline-payload Slot32 table) on the combined int64 key",
                       "inline_probe_batches_per_step": stats["single"]["inline_probes"]},
        "ratio_tuple_over_single": rate["tuple"] / rate["single"],
        "gpu": info, "clocks": clocks}), flush=True)
    if not (check_ok and paths_ok):
        sys.exit(3)


if __name__ == "__main__":
    main()
