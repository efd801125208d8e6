"""Multi-GPU (NCCL) parity tests: sharded groupby with the partial-aggregate exchange and shuffle_table over
all-to-all-v.  Skipped on a machine with one GPU; run on two or more with `python -m pytest tests/test_gpu_multi.py -m gpu`."""

import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    import pandas as pd
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from bodo_b200.shuffle import shuffle_table
        from bodo_b200.streaming.groupby import (delete_groupby_state, groupby_build_consume_batch,
                                                 groupby_produce_output_batch, init_groupby_state)
        from bodo_b200.table import Table
        from oracle import oracle as O
        from tests.helpers import table_to_device
        n_total, n_groups = 600_000, 20_000
        k, v = O.synth_fill(0, n_total, n_groups, 21)
        vf = (v.astype(np.float64) + 0.25)
        chunk = (n_total + world - 1) // world
        lo, hi = rank * chunk, min(n_total, (rank + 1) * chunk)
        df = pd.DataFrame({"k": k[lo:hi], "v": v[lo:hi], "f": vf[lo:hi]})
        t = table_to_device(Table.from_pandas(df), rank)
        # --- sharded groupby: consume local rows in 3 batches, exchange on the last one.  Twice: the fused exchange (pack kernel
        # storing into the owners' slabs over NVLink), then with a slab too small for the partial rows, which must fall back to
        # the NCCL all-to-all-v without losing or double counting anything ---
        fn = ("sum", "count", "mean", "min", "max", "var", "first", "last")
        nloc = hi - lo
        cuts = [0, nloc // 3, 2 * nloc // 3, nloc]
        host = Table.from_pandas(df)
        exp = O.groupby(k, None, list(fn[:5]), [v, v, vf, v, vf], n_pes=world, rank=rank)
        e = pd.DataFrame({"k": exp["keys"], **{f"f{j}": c[0] for j, c in enumerate(exp["cols"])}}).sort_values("k").reset_index(drop=True)
        e["f5"] = pd.DataFrame({"k": k, "vf": vf}).groupby("k").vf.var().reindex(e.k.to_numpy()).to_numpy()  # composite function through the exchange
        # first / last in GLOBAL row order (rank-major: rank r holds rows [r * chunk, (r + 1) * chunk)), carried through the exchange
        gv = pd.DataFrame({"k": k, "v": v}).groupby("k").v
        e["f6"] = gv.first().reindex(e.k.to_numpy()).to_numpy()
        e["f7"] = gv.last().reindex(e.k.to_numpy()).to_numpy()
        ok_keys = ok_int = ok_flt = True
        paths = []
        from bodo_b200.streaming import exchange as X
        for slab_bytes in (None, 8192):
            if slab_bytes is not None:
                os.environ["B200_XCHG_SLAB_BYTES"] = str(slab_bytes)
                X._CACHE.clear()
            st = init_groupby_state(-1, (0,), fn, (0, 1, 2, 3, 4, 5, 6, 7, 8), (1, 1, 2, 1, 2, 2, 1, 1), parallel=True, expected_groups=64, device=rank,
                                    output_batch_size=1 << 30)
            for b in range(3):
                groupby_build_consume_batch(st, table_to_device(host.slice(cuts[b], cuts[b + 1]), rank), b == 2, True)
            out, last = groupby_produce_output_batch(st, True)
            got = out.to_pandas()
            paths.append(st.exchange_path)
            delete_groupby_state(st)
            got.columns = ["k"] + [f"f{j}" for j in range(8)]
            g = got.sort_values("k").reset_index(drop=True)
            okk = bool(len(g) == len(e) and (g.k.to_numpy() == e.k.to_numpy()).all())
            ok_keys = ok_keys and okk
            ok_int = ok_int and okk and all((g[c].to_numpy() == e[c].to_numpy()).all() for c in ("f0", "f1", "f3", "f6", "f7"))
            ok_flt = ok_flt and okk and all(np.allclose(g[c].to_numpy(dtype=float), e[c].to_numpy(dtype=float), rtol=1e-5, atol=1e-8) for c in ("f2", "f4", "f5"))
        os.environ.pop("B200_XCHG_SLAB_BYTES", None)
        X._CACHE.clear()
        ok_keys = ok_keys and paths[1] == "nccl"  # (paths[0] is "fused" wherever symmetric memory is available)
        # --- two-column keys (int64, nullable int32) on the sharded path: fused exchange of multi-key partial rows; every group
        # sits on hash_keys(k0, k1) % world (hash_combine_boost, 4 raw bytes for the int32 column, hash_na_val for NA) ---
        rng2 = np.random.default_rng(5)  # the same global table on every rank
        n2 = 90_000
        a0 = rng2.integers(0, 500, n2).astype(np.int64)
        a1 = rng2.integers(0, 6, n2).astype(np.int32)
        a1v = rng2.random(n2) > 0.15
        w2 = rng2.integers(-50, 50, n2).astype(np.int64)
        gdf = pd.DataFrame({"a0": a0, "a1": pd.array(a1, dtype="Int32"), "w": w2})
        gdf.loc[~a1v, "a1"] = pd.NA
        c2 = (n2 + world - 1) // world
        st2 = init_groupby_state(-1, (0, 1), ("sum", "count", "max"), (0, 1, 2, 3), (2, 2, 2), parallel=True, dropna=False, device=rank,
                                 output_batch_size=1 << 30)
        groupby_build_consume_batch(st2, table_to_device(Table.from_pandas(gdf.iloc[rank * c2:(rank + 1) * c2]), rank), True, True)
        out2, _ = groupby_produce_output_batch(st2, True)
        g2 = out2.to_pandas()
        delete_groupby_state(st2)
        g2.columns = ["a0", "a1", "s", "c", "m"]
        allg = [None] * world
        dist.all_gather_object(allg, g2)
        u = pd.concat(allg, ignore_index=True)
        e2 = gdf.groupby(["a0", "a1"], dropna=False, as_index=False).agg(s=("w", "sum"), c=("w", "count"), m=("w", "max"))
        def canon2(d):
            d = d.copy()
            for c in d.columns:
                d[c] = d[c].to_numpy(dtype="float64", na_value=np.nan)
            return d.sort_values(list(d.columns), na_position="last").reset_index(drop=True)
        ok_mk = bool(canon2(u).shape == canon2(e2).shape and np.array_equal(canon2(u).to_numpy(), canon2(e2).to_numpy(), equal_nan=True))
        # placement: int32 key columns hash their 4 raw bytes -> compare with the reference function through the device helper's
        # oracle-checked twin (tests/test_gpu_shuffle.py pins b200_hash_keys_table against the oracle)
        from bodo_b200.shuffle import hash_keys_table
        if len(g2):
            kt = table_to_device(Table.from_pandas(g2[["a0", "a1"]]), rank)
            _, dest2 = hash_keys_table(kt, 2, world)
            ok_mk = ok_mk and bool((dest2.cpu().numpy() == rank).all())
        ok_keys = ok_keys and ok_mk
        # --- nunique on the sharded path: the nested distinct (key, value) states are exchanged first (pairs owned where the key
        # is owned), then counted into the owned groups ---
        dfu = pd.DataFrame({"k": k[lo:hi], "u": (v[lo:hi] % 7).astype(np.int64)})
        st3 = init_groupby_state(-1, (0,), ("nunique", "count"), (0, 1, 2), (1, 1), parallel=True, device=rank, output_batch_size=1 << 30)
        groupby_build_consume_batch(st3, table_to_device(Table.from_pandas(dfu.iloc[: nloc // 2]), rank), False, True)
        groupby_build_consume_batch(st3, table_to_device(Table.from_pandas(dfu.iloc[nloc // 2:]), rank), True, True)
        out3, _ = groupby_produce_output_batch(st3, True)
        g3 = out3.to_pandas()
        delete_groupby_state(st3)
        g3.columns = ["k", "nu", "c"]
        g3 = g3.sort_values("k").reset_index(drop=True)
        gg = pd.DataFrame({"k": k, "u": v % 7}).groupby("k").u
        owned = e.k.to_numpy()
        ok_nu = bool(len(g3) == len(owned) and (g3.k.to_numpy() == owned).all()
                     and (g3.nu.to_numpy() == gg.nunique().reindex(owned).to_numpy()).all()
                     and (g3.c.to_numpy() == gg.count().reindex(owned).to_numpy()).all())
        ok_keys = ok_keys and ok_nu
        # --- reduce-or-shuffle: nearly unique keys make the ranks switch to the raw-row form (batches are hash-partitioned and
        # exchanged as they come); few groups keep the partial-aggregate form.  Same result either way ---
        os.environ["B200_SHUFFLE_DECISION_ROWS"] = "20000"
        os.environ["B200_COALESCE"] = "0"  # (small batches would sit in the coalescing buffer: nothing to measure yet)
        from bodo_b200.streaming.groupby import get_metric
        modes = []
        for uniq in (True, False):
            rngu = np.random.default_rng(31)
            nu_ = 240_000
            ku = rngu.permutation(nu_).astype(np.int64) if uniq else rngu.integers(0, 300, nu_).astype(np.int64)
            wu = rngu.integers(-9, 9, nu_).astype(np.int64)
            cu = (nu_ + world - 1) // world
            mine = pd.DataFrame({"k": ku[rank * cu:(rank + 1) * cu], "w": wu[rank * cu:(rank + 1) * cu]})
            st4 = init_groupby_state(-1, (0,), ("sum", "count"), (0, 1, 2), (1, 1), parallel=True, device=rank, output_batch_size=1 << 30)
            nb4 = 6
            for b in range(nb4):
                sl = mine.iloc[b * len(mine) // nb4:(b + 1) * len(mine) // nb4]
                groupby_build_consume_batch(st4, Table.from_pandas(sl) if b % 2 else table_to_device(Table.from_pandas(sl), rank), b == nb4 - 1, True)
            modes.append((st4.raw_row_mode, st4.raw_rows_shuffled > 0))
            out4, _ = groupby_produce_output_batch(st4, True)
            g4 = out4.to_pandas()
            delete_groupby_state(st4)
            g4.columns = ["k", "s", "c"]
            allg4 = [None] * world
            dist.all_gather_object(allg4, g4)
            u4 = pd.concat(allg4, ignore_index=True).sort_values("k").reset_index(drop=True)
            e4 = pd.DataFrame({"k": ku, "w": wu}).groupby("k", as_index=False).agg(s=("w", "sum"), c=("w", "count"))
            ok_rs = bool(len(u4) == len(e4) and (u4.to_numpy() == e4.to_numpy()).all())
            ok_place = bool((O.hash_to_rank(g4.k.to_numpy(), None, world) == rank).all())
            if not (ok_rs and ok_place):
                print(f"[rank {rank}] reduce-or-shuffle uniq={uniq}: result ok={ok_rs} placement ok={ok_place} rows {len(u4)} vs {len(e4)}", flush=True)
            ok_keys = ok_keys and ok_rs and ok_place
        if modes != [(True, True), (False, False)] or not ok_nu or not ok_mk:
            print(f"[rank {rank}] modes={modes} ok_nu={ok_nu} ok_mk={ok_mk}", flush=True)
        ok_keys = ok_keys and modes == [(True, True), (False, False)]
        os.environ.pop("B200_SHUFFLE_DECISION_ROWS", None)
        os.environ.pop("B200_COALESCE", None)
        # --- shuffle_table over NCCL: rows land on hash_to_rank(key), nothing lost ---
        sh = shuffle_table(t, 1, True)
        sdf = sh.to_pandas()
        dest = O.hash_to_rank(sdf["k"].to_numpy(), None, world)
        ok_owner = bool((dest == rank).all())
        tot = torch.tensor([len(sdf), int(sdf["v"].sum()), nloc, int(df["v"].sum())], dtype=torch.int64, device=f"cuda:{rank}")
        dist.all_reduce(tot)
        ok_cons = tot[0].item() == tot[2].item() and tot[1].item() == tot[3].item()
        q.put((rank, ok_keys, ok_int, ok_flt, ok_owner, ok_cons, paths))
    except Exception:
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_sharded_groupby_and_shuffle_nccl(gpu_lib):
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=500) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for r in sorted(res, key=lambda x: x[0]):
        assert len(r) == 7 and all(r[1:6]), r
    print("exchange paths per run:", sorted(res, key=lambda x: x[0])[0][6])


def _join_worker(rank, world, port, q):
    import pandas as pd
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from bodo_b200.streaming.join import (delete_join_state, init_join_state, join_build_consume_batch,
                                              join_probe_consume_batch)
        from bodo_b200.table import Table
        from oracle import oracle as O
        rng = np.random.default_rng(77)  # same global tables on every rank; each rank feeds its own row slice
        nb, npr = 40_000, 150_000
        build = pd.DataFrame({"k": rng.integers(0, 30_000, nb).astype(np.int64), "b1": rng.integers(0, 1 << 40, nb),
                              "b2": pd.array(rng.integers(0, 100, nb), dtype="Int64")})
        build.loc[rng.random(nb) < 0.1, "b2"] = pd.NA
        probe = pd.DataFrame({"k": rng.integers(0, 45_000, npr).astype(np.int64), "p1": rng.random(npr)})
        results = {}
        for name, kw, bo, po in (("shuffle", {}, False, False), ("shuffle-outer", {}, True, True),
                                 ("broadcast", {"force_broadcast": True}, False, True)):
            os.environ["BODO_BCAST_JOIN_THRESHOLD"] = "0" if name != "broadcast" else str(10 << 20)  # 0: never broadcast on size
            st = init_join_state(-1, (0,), (0,), tuple(build.columns), tuple(probe.columns), bo, po, build_parallel=True,
                                 probe_parallel=True, device=rank, is_na_equal=True, **kw)
            bchunk, pchunk = (nb + world - 1) // world, (npr + world - 1) // world
            mb = build.iloc[rank * bchunk:(rank + 1) * bchunk]
            mp_ = probe.iloc[rank * pchunk:(rank + 1) * pchunk]
            half = len(mb) // 2
            join_build_consume_batch(st, Table.from_pandas(mb.iloc[:half]), False)
            join_build_consume_batch(st, Table.from_pandas(mb.iloc[half:]), True)
            outs = []
            cuts = [0, len(mp_) // 3, len(mp_)]
            for b in range(2):
                out, _, _ = join_probe_consume_batch(st, Table.from_pandas(mp_.iloc[cuts[b]:cuts[b + 1]]), b == 1, True)
                outs.append(out.to_pandas())
            met = dict(st.metrics)
            delete_join_state(st)
            got = pd.concat(outs, ignore_index=True)
            # global check: gather every rank's output rows, compare the multiset with the oracle join of the global tables
            allg = [None] * world
            dist.all_gather_object(allg, got)
            allm = [None] * world
            dist.all_gather_object(allm, met)
            if rank == 0:
                g = pd.concat(allg, ignore_index=True)
                bi, pi = O.hash_join(build.k.to_numpy(), None, probe.k.to_numpy(), None, bo, po, True)
                def take(df, idx):
                    out = {}
                    for c in df.columns:
                        col = df[c].astype("Float64" if df[c].dtype.kind == "f" else "Int64").take(np.where(idx >= 0, idx, 0)).reset_index(drop=True)
                        col[idx < 0] = pd.NA
                        out[c] = col
                    return out
                e = pd.DataFrame({**{f"b_{c}": v for c, v in take(build, bi).items()}, **{f"p_{c}": v for c, v in take(probe, pi).items()}})
                def canon(df):
                    df = df.copy(); df.columns = [f"c{i}" for i in range(df.shape[1])]
                    for c in df.columns:
                        df[c] = df[c].to_numpy(dtype="float64", na_value=np.nan)
                    return df.sort_values(list(df.columns), na_position="last").reset_index(drop=True)
                cg, ce = canon(g), canon(e)
                ok = cg.shape == ce.shape and bool(np.array_equal(cg.to_numpy(), ce.to_numpy(), equal_nan=True))
                bcast = [m["broadcast"] for m in allm]
                moved = sum(m["build_rows_local"] for m in allm)
                results[name] = (ok, bcast, moved)
                results[name + "/filter"] = ([m.get("filter", 0) for m in allm], sum(m.get("probe_rows_after_filter", 0) for m in allm),
                                             int((pi >= 0).sum() if False else np.isin(probe.k.to_numpy(), build.k.to_numpy()).sum()))
        q.put((rank, results))
    except Exception:
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_sharded_join_shuffle_and_broadcast_nccl(gpu_lib):
    """build_parallel / probe_parallel (bodo/libs/streaming/_join.cpp:3243-3405): rows go to hash_to_rank(key) — or the build side
    is all-gathered (broadcast join) — and the union of the ranks' outputs equals the oracle's join of the global tables."""
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_join_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=500) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    r0 = [r for r in res if r[0] == 0][0]
    assert isinstance(r0[1], dict), r0
    for r in res:
        assert isinstance(r[1], dict), r
    ok, bcast, moved = r0[1]["shuffle"]
    assert ok and bcast == [0] * world and moved == 40_000, r0  # partitioned: every build row lives on exactly one rank
    # inner sharded join: the ranks' bloom filters were OR-ed and applied before the probe shuffle (keys >= 30 000 are outside the
    # build keys' bounds): fewer rows travel, none that has a partner is lost (the join result above is complete)
    flags, after, with_partner = r0[1]["shuffle/filter"]
    assert flags == [1] * world and with_partner <= after < 150_000 * 0.8, r0[1]["shuffle/filter"]
    assert r0[1]["shuffle-outer/filter"][0] == [0] * world  # an outer probe side keeps its rows
    ok, bcast, moved = r0[1]["shuffle-outer"]
    assert ok and bcast == [0] * world, r0
    ok, bcast, moved = r0[1]["broadcast"]
    assert ok and bcast == [1] * world and moved == 40_000 * world, r0  # broadcast: every rank holds the whole build table
