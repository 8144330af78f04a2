"""Cross-shard merge on the GPU, through the C ABI:

* og_query_merge_dense (k_merge_dense) — two shards on one device, merged, against the oracle's scan of the COMBINED shard
  (series of A then series of B: exactly the reference's cross-series update order, reccord_functions.go:47-786).
* og_query_allreduce over the library's own NCCL communicator: world 1 (pack / collectives / fold / CUDA graph on any
  1-GPU box) and world 2 (two processes, two GPUs; skipped when the box has one).

Tolerances: float sums 1e-12 relative (the association differs: (fold A) + (fold B)); everything else bitwise, including the
times carried by min/max/first/last and their tie-breaks.
"""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

import oracle
from opengemini_b200 import AggQuery, Comm, Shard
from opengemini_b200 import _lib as L

pytestmark = pytest.mark.gpu

T0 = 1_700_000_000_000_000_000
SEC = 1_000_000_000
ALL6 = ["count", "sum", "min", "max", "first", "last"]


@pytest.fixture(scope="module", autouse=True)
def _device():
    Shard.init(0)


def _series(seed, n_series, rows, t_shift=0):
    """Coarse values (many ties across series and shards) with a little noise; returns list of arrays."""
    rng = np.random.default_rng(seed)
    return [100.0 + rng.integers(0, 4, rows) * 0.0625 + (rng.random(rows) < 0.05) * rng.random(rows) for _ in range(n_series)]


def _shard(series_values, n=1000, t_first=T0):
    pages, tpages, tmins, tmaxs, ssb = [], [], [], [], [0]
    for v in series_values:
        k = len(v) // n
        for g in range(k):
            pages.append(oracle.field_page_encode(L.TYPE_FLOAT, v[g * n:(g + 1) * n]))
            t = t_first + (np.arange(n, dtype=np.int64) + g * n) * SEC
            tpages.append(oracle.time_page_encode(t)); tmins.append(t[0]); tmaxs.append(t[-1])
        ssb.append(ssb[-1] + k)
    blob, offs, lens, pos = [], [], [], 0
    for p in pages + tpages:
        offs.append(pos); lens.append(p.size); blob.append(p); pos += p.size
    nseg = ssb[-1]
    sh = Shard.open(np.concatenate(blob), np.arange(1, len(series_values) + 1), ssb, tmins, tmaxs,
                    [("v", L.TYPE_FLOAT, offs[:nseg], lens[:nseg])], offs[nseg:], lens[nseg:])
    return sh


def _check(got, ref, calls, label):
    multi = len(calls) > 1
    assert got["n_buckets"] == ref["n_buckets"] and got["start"] == ref["start"], label
    for k, (f, _c) in enumerate(calls):
        gv, rv = got["cols"][k]["valid"].astype(bool), ref["cols"][k]["valid"].astype(bool)
        assert np.array_equal(gv, rv), f"{label} {f}: validity"
        g, r = got["cols"][k]["values"].view(np.uint64)[rv], ref["cols"][k]["values"][rv]
        if f == "sum":
            assert np.allclose(g.view(np.float64), r.view(np.float64), rtol=1e-12, atol=0), f"{label} sum"
        else:
            assert np.array_equal(g, r), f"{label} {f}: values"
        if f in ("min", "max", "first", "last") and not (multi and f in ("min", "max")):
            assert np.array_equal(got["cols"][k]["times"][rv], ref["cols"][k]["times"][rv]), f"{label} {f}: times"


CASES = [[(f, 0)] for f in ALL6] + [[(f, 0) for f in ALL6], [("sum", 0), ("count", 0), ("max", 0)]]


@pytest.mark.parametrize("shifted", [False, True], ids=["same-range", "shifted-range"])
def test_merge_dense_matches_oracle_on_combined_shard(shifted):
    rows = 3000
    a, b = _series(1, 9, rows), _series(2, 5, rows)
    tb = T0 + (1700 * SEC if shifted else 0)  # shard B starts 1700 s later: the shards' own ranges differ -> OG_Q_QUERY_GRID
    sa, sb = _shard(a), _shard(b, t_first=tb)
    tmin, tmax = T0, tb + (rows - 1) * SEC
    # the combined shard the oracle scans: A's series then B's
    ea, eb = sa.export(), sb.export()
    comb = dict(data=np.concatenate([ea["data"], eb["data"]]), sids=np.concatenate([ea["sids"], eb["sids"] + 100]),
                series_seg_begin=np.concatenate([ea["series_seg_begin"], eb["series_seg_begin"][1:] + ea["series_seg_begin"][-1]]),
                seg_tmin=np.concatenate([ea["seg_tmin"], eb["seg_tmin"]]), seg_tmax=np.concatenate([ea["seg_tmax"], eb["seg_tmax"]]),
                col_types=ea["col_types"], page_off=np.concatenate([ea["page_off"], eb["page_off"] + ea["data"].size], axis=1),
                page_len=np.concatenate([ea["page_len"], eb["page_len"]], axis=1))
    sd = oracle.shard_desc_from_export(comb)
    for calls in CASES:
        for iv in (60 * SEC, 7 * SEC, 0):
            qa = AggQuery(sa, calls, iv, tmin, tmax, flags=L.Q_QUERY_GRID | L.Q_STRICT_ORDER).run()
            qb = AggQuery(sb, calls, iv, tmin, tmax, flags=L.Q_QUERY_GRID | L.Q_STRICT_ORDER).run()
            L.check(L.lib().og_query_merge_dense(qa.h, C.byref(qb.dense_view())), "og_query_merge_dense")
            ref = oracle.scan(sd, qa.desc, threads=1)
            _check(qa.dense_host(), ref, calls, f"merge_dense {calls} iv={iv}")
            qa.close(); qb.close()
    if shifted:  # without the common grid the merge must refuse, not mis-align buckets
        qa = AggQuery(sa, [("sum", 0)], 60 * SEC, tmin, tmax).run()
        qb = AggQuery(sb, [("sum", 0)], 60 * SEC, tmin, tmax).run()
        assert L.lib().og_query_merge_dense(qa.h, C.byref(qb.dense_view())) == L.OG_E_INVAL
        qa.close(); qb.close()
    sa.close(); sb.close()


def test_allreduce_world1_is_identity_and_replays_its_graph():
    rows = 4000
    sh = _shard(_series(3, 40, rows))
    comm = Comm.init_rank(Comm.unique_id(), 0, 1)
    assert comm.info()["world"] == 1
    for calls in CASES:
        q = AggQuery(sh, calls, 60 * SEC, T0, T0 + (rows - 1) * SEC, flags=L.Q_QUERY_GRID).run()
        before = q.dense_host()
        for _ in range(3):  # first call captures the graph, the next ones replay it
            comm.allreduce(q)
            after = q.dense_host()
            for k in range(len(calls)):
                m = before["cols"][k]["valid"].astype(bool)
                assert np.array_equal(after["cols"][k]["valid"].astype(bool), m)
                assert np.array_equal(after["cols"][k]["values"].view(np.uint64)[m], before["cols"][k]["values"].view(np.uint64)[m])
                if before["cols"][k]["times"] is not None:
                    assert np.array_equal(after["cols"][k]["times"][m], before["cols"][k]["times"][m])
        assert q.stats()["merge_ms"] > 0
        q.close()
    comm.close(); sh.close()


def _rank_main(rank, world, idfile, out):
    import time
    from opengemini_b200 import _lib as L2
    Shard.init(rank)
    if rank == 0:
        uid = Comm.unique_id()
        with open(idfile + ".tmp", "wb") as f:
            f.write(uid)
        os.replace(idfile + ".tmp", idfile)
    else:
        for _ in range(600):
            if os.path.exists(idfile):
                break
            time.sleep(0.05)
        uid = open(idfile, "rb").read()
    comm = Comm.init_rank(uid, rank, world)
    rows = 3000
    sh = _shard(_series(10 + rank, 6 + rank, rows), t_first=T0 + rank * 1300 * SEC)
    res = {}
    for ci, calls in enumerate(CASES):
        q = AggQuery(sh, calls, 60 * SEC, T0, T0 + 1300 * SEC * (world - 1) + (rows - 1) * SEC, flags=L2.Q_QUERY_GRID | L2.Q_STRICT_ORDER).run()
        comm.allreduce(q)
        d = q.dense_host()
        res[ci] = [(c["values"].view(np.uint64).copy(), c["valid"].copy(), None if c["times"] is None else c["times"].copy()) for c in d["cols"]]
        res[(ci, "geom")] = (d["n_buckets"], d["start"])
        q.close()
    comm.close(); sh.close()
    out.put((rank, res))


def test_allreduce_two_gpus_matches_oracle():
    if L.lib().og_device_count() < 2:
        pytest.skip("needs two GPUs")
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    world = 2
    with tempfile.TemporaryDirectory() as td:
        idfile = os.path.join(td, "nccl_id")
        procs = [ctx.Process(target=_rank_main, args=(r, world, idfile, out)) for r in range(world)]
        for p in procs:
            p.start()
        got = dict(out.get(timeout=300) for _ in range(world))
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    rows = 3000
    shards = [_shard(_series(10 + r, 6 + r, rows), t_first=T0 + r * 1300 * SEC) for r in range(world)]
    exs = [s.export() for s in shards]
    comb = dict(data=np.concatenate([e["data"] for e in exs]), sids=np.concatenate([e["sids"] + 100 * i for i, e in enumerate(exs)]),
                series_seg_begin=np.concatenate([exs[0]["series_seg_begin"], exs[1]["series_seg_begin"][1:] + exs[0]["series_seg_begin"][-1]]),
                seg_tmin=np.concatenate([e["seg_tmin"] for e in exs]), seg_tmax=np.concatenate([e["seg_tmax"] for e in exs]),
                col_types=exs[0]["col_types"], page_off=np.concatenate([exs[0]["page_off"], exs[1]["page_off"] + exs[0]["data"].size], axis=1),
                page_len=np.concatenate([e["page_len"] for e in exs], axis=1))
    sd = oracle.shard_desc_from_export(comb)
    tmax = T0 + 1300 * SEC * (world - 1) + (rows - 1) * SEC
    for ci, calls in enumerate(CASES):
        q = AggQuery(shards[0], calls, 60 * SEC, T0, tmax, flags=L.Q_QUERY_GRID)
        ref = oracle.scan(sd, q.desc, threads=1)
        q.close()
        for r in range(world):
            cols = [dict(values=v.view(np.float64), valid=k, times=t) for v, k, t in got[r][ci]]
            g = dict(n_buckets=got[r][(ci, "geom")][0], start=got[r][(ci, "geom")][1], cols=cols)
            _check(g, ref, calls, f"allreduce rank {r} {calls}")
        for k in range(len(calls)):  # every rank holds the same bits
            assert np.array_equal(got[0][ci][k][0], got[1][ci][k][0]) and np.array_equal(got[0][ci][k][1], got[1][ci][k][1])
    for s in shards:
        s.close()
