#!/usr/bin/env python
"""bench.py — decoded+aggregated rows/s of the fused scan/aggregate path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          # our arm (libogpu.so, sm_100a kernels)
    python bench.py --impl reference --gpus N ...          # reference arm: the CPU oracle on the host cores

Workload (config.workload): BASELINE.json configs[1] — one TSM shard of 10k series x 1M points/series of float64
(G-hi distribution: 100 + U[0,1) with full mantissa tail -> Gorilla ~6 B/value), 1 s cadence, const-delta time pages,
1000-row segments; SELECT sum, count (mean) and max GROUP BY time(1m), all series in one tagset.
A "step" = one og_query_run over the whole HBM-resident shard (k_fused_fast over the lane-interleaved Gorilla streams, k_fused_raw for raw pages, edge stitch + tagset
merge).  At N > 1 every rank holds its own shard (distinct seed; configs[3]) and a step ends with the NCCL
cross-shard merge of the dense bucket arrays (weak scaling).

The JSON line follows the driver contract; `roofline` is the fused kernel alone, `e2e` goes through the C ABI with
host buffers (og_shard_open H2D + query + og_query_next D2H inside the timed region), `cpu_baseline` is the oracle.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

T0, SEC = 1_700_000_000_000_000_000, 1_000_000_000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--series", type=int, default=10_000)
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--dist", default="hi", choices=["hi", "lo"])
    ap.add_argument("--e2e-series", type=int, default=2000, help="series of the host-resident sample used by the e2e leg")
    ap.add_argument("--cpu-series", type=int, default=0, help="series of the CPU sample (0 = auto: 4 per host thread)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--workload", default="float", choices=["float", "mixed", "downsample"],
                    help="float = configs[1] (the headline, default); mixed = configs[2]: int64 Simple8b + float64 Gorilla + bool columns, "
                         "count(i), sum(i), sum(f), count(b) WHERE f > 1000 GROUP BY time(1m) (a secondary line with its own roofline)")
    ap.add_argument("--nulls", type=int, default=0, help="mixed workload: null permille of every column (50 = the 5 %% variant)")
    ap.add_argument("--no-verify", action="store_true", help="skip the answer check after the timed loop")
    ap.add_argument("--verify-series", type=int, default=4, help="series sampled for the bitwise check against the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the arrays the last step returned as DIR/<name>.npy "
                                                          "(float64 / float32, at most 64 MB in all) to compare two builds output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path returned: it needs --impl ours")
    return a


DUMP_LIMIT = 60_000_000  # bytes of array data: the files stay under 64 MB with their .npy headers


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """Write {name: array} as out_dir/<name>.npy.  Integers and float64 go out as float64 (an integer that float64 cannot hold
    exactly is an error: times are passed as offsets from T0), bytes and flags as float32.  While the whole exceeds `limit`, the
    largest array is replaced by its elements at sorted positions drawn with a fixed seed; the positions go to <name>_index.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        a = np.ascontiguousarray(a).ravel()
        f = a.astype(np.float32 if a.dtype.itemsize <= 2 else np.float64)
        if a.dtype.kind in "iub" and not np.array_equal(f.astype(a.dtype), a):
            raise ValueError(f"--dump-outputs: {name} holds integers that {f.dtype} cannot represent exactly")
        out[name] = f
    while sum(v.nbytes for v in out.values()) > limit:
        name = max((k for k in arrays if k + "_index" not in out), key=lambda k: out[k].nbytes)
        v = out[name]
        room = limit - (sum(x.nbytes for x in out.values()) - v.nbytes)
        m = max(1, room // (v.itemsize + 8))
        idx = np.sort(np.random.default_rng(0).choice(v.size, size=min(m, v.size - 1), replace=False))
        out[name], out[name + "_index"] = v[idx], idx.astype(np.float64)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def dense_arrays(d, calls):
    """The dense interval record a query returns (AggQuery.dense_host()), one array per field; times relative to T0."""
    import numpy as np
    arrays = {"grid": np.array([d["n_groups"], d["n_buckets"], d["start"] - T0, d["interval"]], np.int64)}
    for (func, col), c in zip(calls, d["cols"]):
        arrays[f"{func}_f{col}_values"] = c["values"]
        arrays[f"{func}_f{col}_valid"] = c["valid"]
        if c["times"] is not None:
            arrays[f"{func}_f{col}_times"] = c["times"] - T0
    return arrays


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe), in-process through NVML
    (a background thread; og_query_run releases the GIL), falling back to one nvidia-smi query when NVML is missing."""

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.t, self.h = index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
        except Exception:
            self.h = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, mx, rs))
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        if self.h is not None:
            self.stop_flag = True
            self.t.join(timeout=2)
            if not self.rows:
                self._poll_once()
            sm = sorted(r[0] for r in self.rows)
            reasons = sorted({n for r in self.rows for bit, n in names.items() if r[2] & bit})
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((r[1] for r in self.rows), default=None),
                    "reasons": reasons, "samples": len(sm), "source": "nvml"}
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=10).stdout.split(",")
            return {"sm_mhz": int(float(out[0])), "sm_max_mhz": int(float(out[1])), "reasons": [], "samples": 1, "source": "nvidia-smi after the region"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"], "samples": 0}

    def _poll_once(self):
        self.stop_flag = True
        try:
            nv = self.nv
            self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM), 0))
        except Exception:
            pass


def ncu_traffic(a):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu --set full capture
    (profiles/traffic.json); only valid for the workload it was captured on, else null."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if a.workload == "mixed":
            if a.series == 10000 and a.rows == 1000000 and a.nulls == 0:  # the mixed workload's own defaults (50k x 20k) are substituted for these
                return t["k_fused_cols"]["dram_bytes_per_launch"]
        elif a.series == 10000 and a.rows == 1000000 and a.dist == "hi":
            return t["k_fused_il"]["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


def measured_peak():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def workload_name(a):
    return (f"configs[1]: {a.series} series x {a.rows} float64 points/series, G-{a.dist} (Gorilla), 1s cadence, 1000-row segments, "
            f"sum+count(mean)+max GROUP BY time(1m), one tagset")


def dist_const(L, a):
    return L.SYNTH_F_HI if a.dist == "hi" else L.SYNTH_F_LO


# ---------------------------------------------------------------------------------------------------------------
# reference arm: the reference's algorithm on the host cores (the Go engine cannot be built in this image: the
# oracle is its C++ restatement, see oracle/og_oracle.h)
# ---------------------------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU arm can really use: hardware threads visible to this process, capped by the container's CPU quota
    (cgroup cpu.max) — on the graft B200 boxes nproc says 128 but the quota is 16 CPUs, and running 128 threads under a
    16-CPU quota is slower than 16-32.  Returns (candidate thread counts, note)."""
    hw = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = max(1, int(round(int(q) / int(per))))
    except Exception:
        pass
    if quota is None or quota >= hw:
        return [hw], f"{hw} hardware threads, no cgroup quota"
    return sorted({min(hw, quota), min(hw, 2 * quota)}), f"{hw} hardware threads, cgroup cpu.max quota = {quota} CPUs"


def best_threads(L, a, hs, qd, cands):
    """One short scan per candidate thread count; keep the fastest."""
    import oracle
    best, best_v = cands[0], 0.0
    if len(cands) == 1:
        return best
    for th in cands:
        t0 = time.perf_counter()
        oracle.scan(hs.desc, qd, threads=th, fast=True)
        v = 1.0 / (time.perf_counter() - t0)
        if v > best_v:
            best, best_v = th, v
    return best


def cpu_sample(L, a, n_series, threads):
    import oracle
    hs = oracle.HostShard(n_series, a.rows, [(L.TYPE_FLOAT, dist_const(L, a), 0)], t0=T0, dt=SEC, seed=1000, threads=threads)
    return hs


def query_desc(L, a):
    calls = (L.Call * 3)()
    for i, f in enumerate((L.AGG_SUM, L.AGG_COUNT, L.AGG_MAX)):
        calls[i].func, calls[i].column = f, 0
    d = L.QueryDesc()
    d.interval, d.offset, d.tmin, d.tmax, d.ascending = 60 * SEC, 0, T0, T0 + (a.rows - 1) * SEC, 1
    d.n_calls, d.calls, d.n_filter, d.group_mode, d.chunk_size = 3, calls, 0, L.GROUP_ALL, 1024
    d._keep = calls
    return d


def run_reference(a):
    from opengemini_b200 import _lib as L
    import oracle
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cands, note = host_threads()
    n = a.cpu_series or min(a.series, 32 * cands[-1], 2048)
    hs = cpu_sample(L, a, n, cands[-1])
    qd = query_desc(L, a)
    threads = best_threads(L, a, hs, qd, cands)
    rows = n * a.rows
    for _ in range(a.warmup):
        oracle.scan(hs.desc, qd, threads=threads, fast=True)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        r = oracle.scan(hs.desc, qd, threads=threads, fast=True)
    dt = time.perf_counter() - t0
    v = rows * a.steps / dt
    line = {"impl": "reference", "metric": "decoded+aggregated rows/s", "value": v, "unit": "rows/s", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": {"workload": workload_name(a), "sample": f"{n} series x {a.rows} rows per step"},
            "cpu_baseline": {"value": v, "unit": "rows/s", "cores": threads, "kind": "port",
                             "sample": f"{n} series x {a.rows} rows ({rows} rows, {r['page_bytes']} page bytes) per step; C++ restatement of the reference pull loop with its batch "
                                       f"Gorilla decoder (64-bit cached bit reader, batch_float.go:308-347; oracle/fast_scan.cpp, checked against the oracle); " + note},
            "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
class VerifyError(RuntimeError):
    pass


def verify_answer(a, L, sh, q, calls, tmax, rank, info):
    """The timed query's answer, checked at full size (the run fails with rc != 0 on a mismatch):
    (1) sum of the per-bucket counts == rows of the shard;
    (2) the folded (default) sums against the strict-order run of the same query: <= 1e-12 relative; counts and max bitwise;
    (3) K sampled series, aggregated on the GPU through a tag-group map (strict per-series order), bitwise against the CPU
        oracle's scan of the same series rebuilt from the same seed (og_synth_desc.series_base)."""
    import numpy as np
    import oracle
    from opengemini_b200 import AggQuery
    t0 = time.perf_counter()
    q.run()  # this shard's own answer (at N > 1 the timed steps left the cross-shard merge in the dense arrays)
    d = q.dense_host()
    cnt = d["cols"][1]["values"].astype(np.int64) * d["cols"][1]["valid"]
    if int(cnt.sum()) != int(info["n_rows"]):
        raise VerifyError(f"sum of bucket counts {int(cnt.sum())} != rows {info['n_rows']}")
    qs = AggQuery(sh, calls, 60 * SEC, T0, tmax, flags=L.Q_STRICT_ORDER).run()
    ds = qs.dense_host()
    qs.close()
    for k, name in enumerate(("sum", "count", "max")):
        if not np.array_equal(d["cols"][k]["valid"], ds["cols"][k]["valid"]):
            raise VerifyError(f"{name}: validity of the folded and the strict-order run differ")
        m = ds["cols"][k]["valid"].astype(bool)
        if name == "sum":
            rel = np.abs(d["cols"][k]["values"][m] - ds["cols"][k]["values"][m]) / np.abs(ds["cols"][k]["values"][m])
            if rel.size and rel.max() > 1e-12:
                raise VerifyError(f"folded sums differ from strict-order sums by {rel.max():.3e} relative")
            max_rel = float(rel.max()) if rel.size else 0.0
        elif not np.array_equal(d["cols"][k]["values"].view(np.uint64)[m], ds["cols"][k]["values"].view(np.uint64)[m]):
            raise VerifyError(f"{name}: folded and strict-order runs differ")
    K = max(0, min(a.verify_series, a.series))
    rng = np.random.default_rng(12345 + rank)
    picks = sorted(set(int(x) for x in rng.integers(0, a.series, K))) if K else []
    if picks:
        grp = np.zeros(a.series, np.uint32)
        for i, s_ in enumerate(picks):
            grp[s_] = i + 1
        qm = AggQuery(sh, calls, 60 * SEC, T0, tmax, group="map", series_group=grp, n_groups=len(picks) + 1).run()
        dm = qm.dense_host()
        nb = dm["n_buckets"]
        for i, s_ in enumerate(picks):
            hs = oracle.HostShard(1, a.rows, [(L.TYPE_FLOAT, dist_const(L, a), 0)], t0=T0, dt=SEC, seed=1000 + rank, series_base=s_)
            ref = oracle.scan(hs.desc, q.desc, threads=1)
            for k, name in enumerate(("sum", "count", "max")):
                gv = dm["cols"][k]["valid"][(i + 1) * nb:(i + 2) * nb].astype(bool)
                gb = dm["cols"][k]["values"].view(np.uint64)[(i + 1) * nb:(i + 2) * nb]
                rv = ref["cols"][k]["valid"].astype(bool)
                if not np.array_equal(gv, rv) or not np.array_equal(gb[rv], ref["cols"][k]["values"][rv]):
                    raise VerifyError(f"series {s_}: {name} differs from the oracle (bitwise)")
        qm.close()
    return {"rows_counted": int(cnt.sum()), "folded_vs_strict_sum_max_rel": max_rel, "series_checked_bitwise_vs_oracle": picks,
            "seconds": round(time.perf_counter() - t0, 2)}

def make_comm(torch, dist, Comm, rank, world, dev):
    """The library's own NCCL communicator (og_comm_*): rank 0's 128-byte id travels over torch.distributed (plumbing only);
    the merge itself is og_query_allreduce inside libogpu.so."""
    idt = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        idt.copy_(torch.frombuffer(bytearray(Comm.unique_id()), dtype=torch.uint8))
    dist.broadcast(idt, src=0)
    return Comm.init_rank(bytes(idt.cpu().numpy().tobytes()), rank, world)


def verify_merge(a, L, comm, rank, world):
    """configs[3] answer check at N > 1: every rank builds a SMALL shard (own seed), runs the bench query and the library's
    NCCL merge; the merged record (identical on every rank) is compared with the oracle's scans of the same shards merged on the
    host with the reference's rules (sum/count add, max = larger).  Sums 1e-9 relative, counts and max exact."""
    import numpy as np
    import oracle
    from opengemini_b200 import AggQuery, Shard
    ns, rows = 64, 20_000
    cols = [(L.TYPE_FLOAT, dist_const(L, a), 0)]
    calls = [("sum", 0), ("count", 0), ("max", 0)]
    sh = Shard.synth(ns, rows, cols, t0=T0, dt=SEC, seed=7000 + rank)
    q = AggQuery(sh, calls, 60 * SEC, T0, T0 + (rows - 1) * SEC, flags=L.Q_QUERY_GRID).run()
    comm.allreduce(q)
    got = q.dense_host()
    exp = None
    for r in range(world):
        hs = oracle.HostShard(ns, rows, cols, t0=T0, dt=SEC, seed=7000 + r)
        ref = oracle.scan(hs.desc, q.desc, threads=1)
        part = [(c["values"].copy(), c["valid"].astype(bool)) for c in ref["cols"]]
        if exp is None:
            exp = part
            continue
        (s0, k0), (c0, kc0), (m0, km0) = exp
        (s1, k1), (c1, kc1), (m1, km1) = part
        ssum = np.where(k0, s0.view(np.float64), 0.0) + np.where(k1, s1.view(np.float64), 0.0)
        cnt = np.where(kc0, c0.view(np.int64), 0) + np.where(kc1, c1.view(np.int64), 0)
        mx = np.where(km0 & km1, np.maximum(m0.view(np.float64), m1.view(np.float64)), np.where(km0, m0.view(np.float64), m1.view(np.float64)))
        exp = [(ssum.view(np.uint64), k0 | k1), (cnt.view(np.uint64), kc0 | kc1), (mx.view(np.uint64), km0 | km1)]
    for k, name in enumerate(("sum", "count", "max")):
        ev, ek = exp[k]
        if not np.array_equal(got["cols"][k]["valid"].astype(bool), ek):
            raise VerifyError(f"merged {name}: validity differs from the oracle")
        g = got["cols"][k]["values"]
        if name == "sum":
            rel = np.abs(g[ek] - ev.view(np.float64)[ek]) / np.abs(ev.view(np.float64)[ek])
            if rel.max() > 1e-9:
                raise VerifyError(f"merged sums off by {rel.max():.3e} relative")
        elif not np.array_equal(g.view(np.uint64)[ek], ev[ek]):
            raise VerifyError(f"merged {name} differs from the oracle")
    q.close(); sh.close()
    return {"shards": world, "series_per_shard": ns, "rows_per_series": rows, "checked": "sum<=1e-9 rel, count and max exact vs the oracle on the same shards"}


def run_ours(a):
    import numpy as np
    import torch
    from opengemini_b200 import AggQuery, Comm, Shard
    from opengemini_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the communicator is created; stdout must carry the JSON line only
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            warm = torch.zeros(1, device=torch.device("cuda", local))
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    Shard.init(local)
    dev = torch.device("cuda", local)
    cols = [(L.TYPE_FLOAT, dist_const(L, a), 0)]
    t_gen = time.perf_counter()
    sh = Shard.synth(a.series, a.rows, cols, t0=T0, dt=SEC, seed=1000 + rank)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t_gen
    info = sh.info()
    calls = [("sum", 0), ("count", 0), ("max", 0)]
    tmax = T0 + (a.rows - 1) * SEC
    comm = make_comm(torch, dist, Comm, rank, world, dev) if world > 1 else None
    q = AggQuery(sh, calls, 60 * SEC, T0, tmax, flags=L.Q_QUERY_GRID if world > 1 else 0)
    merge_ms_total = [0.0]

    def step():
        q.run()
        st = q.stats()
        ms = st["kernel_ms"]
        if comm is not None:  # cross-shard merge inside libogpu.so (NCCL all-reduce + all-gather/fold, one CUDA graph); CUDA events on the query stream
            comm.allreduce(q)
            m = q.stats()["merge_ms"]
            ms += m
            merge_ms_total[0] += m
        return ms, st

    for _ in range(max(a.warmup, 3)):
        step()
    sampler = ClockSampler(local)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    dev_ms, main_ms, launches = 0.0, 0.0, 0
    for _ in range(a.steps):
        ms, st = step()
        dev_ms += ms
        main_ms += st["main_kernel_ms"]
        launches += st["kernel_launches"]
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall_s = time.perf_counter() - w0
    clocks = sampler.stop()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, dense_arrays(q.dense_host(), calls))
    t = torch.tensor([dev_ms, wall_s * 1e3], dtype=torch.float64, device=dev)
    rows_t = torch.tensor([float(st["rows_decoded"])], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(rows_t, op=dist.ReduceOp.SUM)
    dev_ms_max, wall_ms_max = t.tolist()
    total_rows = rows_t.item()
    value = total_rows * a.steps / (dev_ms_max / 1e3)

    # warm end-to-end: the shard stays resident in HBM (the deployment this library is built for: a shard is uploaded once and
    # queried many times); a step = og_query_run + draining og_query_next into host records
    resident = None
    if not a.no_e2e:
        r_steps = max(1, min(a.steps, 5))
        torch.cuda.synchronize()
        tr0 = time.perf_counter()
        for _ in range(r_steps):
            q.run()
            if comm is not None:
                comm.allreduce(q)
            out_rows_r = sum(rec["rows"] for rec in q.records())
        tr = time.perf_counter() - tr0
        resident = {"value": float(info["n_rows"]) * world * r_steps / tr, "unit": "rows/s", "ms_per_step": tr / r_steps * 1e3, "steps": r_steps, "out_rows": out_rows_r,
                    "what": "og_query_run + og_query_next until OG_EOF on the HBM-resident shard (host wall clock, D2H of the result inside)"}
    verify = verify_answer(a, L, sh, q, calls, tmax, rank, info) if not a.no_verify else None
    if comm is not None and not a.no_verify:
        vm = verify_merge(a, L, comm, rank, world)
        if verify is not None:
            verify["cross_shard_merge"] = vm

    # roofline of the dominant kernel: algorithmic bytes per launch / its average duration
    peak, peak_src = measured_peak()
    algo_bytes = st["page_bytes"] + st["dir_bytes"] + st["out_bytes"]  # pages + 32 B/segment directory + dense output (og_stats)
    main_per_launch_ms = main_ms / a.steps
    achieved = algo_bytes / (main_per_launch_ms / 1e3) / 1e9
    kernel_name = {3: "k_fused_il<SUM|COUNT|MAX, fold> (+ k_fused_segment for %d general segments)" % st["general_segments"],
                   2: "k_fused_il<SUM|COUNT|MAX> (+ k_fused_segment)", 1: "k_fused_segment", 0: "k_decode_tile+k_filter_tile+k_window_reduce"}[st["path"]]
    roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(a), "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes,
                "bytes_per_row": algo_bytes / max(1, st["rows_decoded"]), "kernel_ms": main_per_launch_ms,
                "share_of_step": main_ms / max(1e-9, dev_ms if world == 1 else main_ms),
                "interleaved_copy": {"build_ms_once_per_shard": st["il_build_ms"], "bytes": st["il_bytes"], "state": st["il_state"],
                                     "note": "built by the first query on the column (inside warm-up here, inside the timed region of the e2e leg)"}}

    # e2e: the call a user of the C ABI makes, with HOST buffers (pinned), H2D + query + D2H in the timed region
    e2e = None
    e2e_launches = 0
    # the HBM-resident shard of the timed region is released first: the e2e leg measures a cold open of its own shard and should
    # not depend on how much device memory the first leg left allocated
    q.close()
    sh.close()
    q = sh = None
    if not a.no_e2e:
        ns = min(a.e2e_series, a.series)
        small = Shard.synth(ns, a.rows, cols, t0=T0, dt=SEC, seed=1000 + rank)
        lay = L.ShardLayout()
        L.check(L.lib().og_shard_layout_get(small.h, C.byref(lay)), "layout")
        pinned = torch.empty(lay.data_len, dtype=torch.uint8, pin_memory=True)
        ex = dict(sids=np.empty(ns, np.uint64), series_seg_begin=np.empty(ns + 1, np.uint32), seg_tmin=np.empty(lay.n_segments, np.int64),
                  seg_tmax=np.empty(lay.n_segments, np.int64), page_off=np.empty((2, lay.n_segments), np.uint64),
                  page_len=np.empty((2, lay.n_segments), np.uint32), col_types=np.empty(1, np.int32))
        L.check(L.lib().og_shard_export(small.h, pinned.data_ptr(), *[ex[k].ctypes.data for k in
                                                                        ("sids", "series_seg_begin", "seg_tmin", "seg_tmax", "page_off", "page_len", "col_types")]), "export")
        small.close()
        host_data = pinned.numpy()
        h2d = int(lay.data_len + lay.n_segments * (2 * 12 + 16) + ns * 12)
        e_steps = max(1, min(a.steps, 3))

        phases = {"open": 0.0, "query": 0.0, "records": 0.0, "close": 0.0}

        def e2e_step():
            p0 = time.perf_counter()
            s2 = Shard.open(host_data, ex["sids"], ex["series_seg_begin"], ex["seg_tmin"], ex["seg_tmax"],
                            [("f0", L.TYPE_FLOAT, ex["page_off"][0], ex["page_len"][0])], ex["page_off"][1], ex["page_len"][1])
            p1 = time.perf_counter()
            q2 = AggQuery(s2, calls, 60 * SEC, T0, tmax).run()
            p2 = time.perf_counter()
            out_rows, d2h = 0, 0
            for rec in q2.records():
                out_rows += rec["rows"]
                d2h += sum(c["values"].nbytes + (c["len"] + 7) // 8 for c in rec["cols"]) + rec["times"].nbytes
            ln = q2.stats()["kernel_launches"] + 2
            p3 = time.perf_counter()
            q2.close(); s2.close()
            p4 = time.perf_counter()
            for k, v in zip(("open", "query", "records", "close"), (p1 - p0, p2 - p1, p3 - p2, p4 - p3)):
                phases[k] += v * 1e3
            return out_rows, d2h, ln

        e2e_step()
        for k in phases:
            phases[k] = 0.0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            out_rows, d2h, ln = e2e_step()
            e2e_launches += ln
        torch.cuda.synchronize()
        et = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(et, op=dist.ReduceOp.MAX)
        e_rows = ns * a.rows * world
        # d2h: the three dense columns (value + validity) are copied back whole before records are sliced
        d2h_full = int(st["out_bytes"])
        e2e = {"value": e_rows * e_steps / et.item(), "unit": "rows/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": max(d2h, d2h_full),
               "sample": f"{ns} series x {a.rows} rows per GPU per step (host-resident, pinned), og_shard_open + og_query_run + og_query_next",
               "resident": resident,
               "sample_note": "2000 of the 10000 series per step: pinning and re-uploading the full 61 GB shard every step would take minutes; rates, not totals, are compared",
               "steps": e_steps, "phase_ms_per_step": {k: round(v / e_steps, 2) for k, v in phases.items()}, "ms_per_step": et.item() / e_steps * 1e3, "out_rows": out_rows}
        # the cold path is the host-to-device copy: og_shard_open is one blocking copy of the pages plus the directory
        open_s = phases.get("open", 0.0) / e_steps / 1e3
        if open_s > 0:
            e2e["h2d_GBps_inside_open"] = h2d / open_s / 1e9
            e2e["copy_share_of_step"] = open_s / (et.item() / e_steps)
            e2e["bound"] = "PCIe: with the copy alone the step could not exceed %.2f G rows/s" % (ns * a.rows / open_s / 1e9)
        del pinned

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        import oracle
        cands, note = host_threads()
        n = a.cpu_series or min(a.series, 32 * cands[-1], 2048)
        hs = cpu_sample(L, a, n, cands[-1])
        qd = query_desc(L, a)
        threads = best_threads(L, a, hs, qd, cands)  # also warms
        reps, t0 = 0, time.perf_counter()
        while True:
            r = oracle.scan(hs.desc, qd, threads=threads, fast=True)
            reps += 1
            el = time.perf_counter() - t0
            if el > 8 or reps >= 20:
                break
        t1 = time.perf_counter()
        r1 = oracle.scan(hs.desc, qd, threads=1, s1=1, fast=True)
        one = a.rows / (time.perf_counter() - t1)
        t2 = time.perf_counter()
        oracle.scan(hs.desc, qd, threads=1, s1=1)
        checker_one = a.rows / (time.perf_counter() - t2)
        cpu = {"value": n * a.rows * reps / el, "unit": "rows/s", "cores": threads, "kind": "port",
               "sample": f"{n} series x {a.rows} rows x {reps} repetitions in {el:.1f}s; C++ restatement of the reference pull loop "
                         f"(batch Gorilla decode with a 64-bit cached bit reader -> FilterByTime -> window reduce -> AggTagSet merge; oracle/fast_scan.cpp), "
                         f"series strided over {threads} threads; {note}",
               "single_thread_rows_per_s": one, "decoded_MBps_per_thread": one * 8 / 1e6,
               "reference_reported_MBps_per_core": "320-340 (batch_float.go:303-306, 2016 laptop)",
               "bit_serial_checker_rows_per_s_single_thread": checker_one}
        del r1

    if rank == 0:
        line = {"metric": "decoded+aggregated rows/s", "value": value, "unit": "rows/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
                "ms_per_step": dev_ms_max / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "impl": "ours",
                "config": {"workload": workload_name(a), "shards": world, "rows_per_shard": int(info["n_rows"]), "segments_per_shard": int(info["n_segments"]),
                           "page_bytes_per_shard": int(info["page_bytes"]), "compressed_bytes_per_value": info["page_bytes"] / max(1, info["n_rows"]),
                           "l2": "inputs (tens of GB per step) are far larger than the 126 MB L2; no explicit flush",
                           "parallelism": f"shard-per-gpu x{world}" + (", og_query_allreduce: NCCL all-reduce(sum,count) + all-gather/fold(max) inside libogpu.so" if world > 1 else ""),
                           "timing": "CUDA events on the query stream (og_stats.kernel_ms + og_stats.merge_ms); max over ranks",
                           "merge_ms_per_step": merge_ms_total[0] / (max(a.warmup, 3) + a.steps) if world > 1 else 0.0,
                           "synth_seconds": gen_s},
                "wall_ms_per_step": wall_ms_max / a.steps, "clocks": clocks, "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu, "verify": verify,
                "gpu_launches": launches + e2e_launches}
        print(json.dumps(line), flush=True)
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def run_mixed(a):
    """configs[2] on one GPU: 50k series x 20k rows (10^9 rows) of int64 (Simple8b) + float64 (Gorilla, G-lo) + bool columns,
    count(i), sum(i), sum(f), count(b) WHERE f > 1000 GROUP BY time(1m); --nulls 50 = the 5 % nulls variant.  One step = one
    og_query_run (k_fused_cols: one thread per segment walks one column at a time in a codec-specialised loop, columns meet through
    a per-thread row mask; nothing materialised.  OGPU_NO_COLS=1 selects the older pull-iterator kernel k_fused_multi).  The answer is checked against the oracle
    on a slice of the same synthetic population (series_base)."""
    import numpy as np
    import torch
    import oracle
    from opengemini_b200 import AggQuery, Shard
    from opengemini_b200 import _lib as L
    torch.cuda.set_device(0)
    Shard.init(0)
    series = a.series if a.series != 10_000 else 50_000
    rows = a.rows if a.rows != 1_000_000 else 20_000
    cols = [(L.TYPE_INT, L.SYNTH_INT_WALK, a.nulls), (L.TYPE_FLOAT, L.SYNTH_F_LO, a.nulls), (L.TYPE_BOOL, L.SYNTH_BOOL, a.nulls)]
    sh = Shard.synth(series, rows, cols, t0=T0, dt=SEC, seed=4242)
    info = sh.info()
    calls = [("count", 0), ("sum", 0), ("sum", 1), ("count", 2)]
    flt = [("term", 1, ">", 1000.0)]
    tmax = T0 + (rows - 1) * SEC
    q = AggQuery(sh, calls, 60 * SEC, T0, tmax, filter=flt)
    for _ in range(max(a.warmup, 3)):
        q.run()
    sampler = ClockSampler(0); sampler.start()
    dev_ms = main_ms = 0.0; launches = 0
    for _ in range(a.steps):
        q.run(); st = q.stats()
        dev_ms += st["kernel_ms"]; main_ms += st["main_kernel_ms"]; launches += st["kernel_launches"]
    clocks = sampler.stop()
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, dense_arrays(q.dense_host(), calls))
    # answer check on a slice: the first K series of the population, same seed, through the oracle
    verify = None
    if not a.no_verify:
        K = min(series, 64)
        small = Shard.synth(K, rows, cols, t0=T0, dt=SEC, seed=4242)
        hs = oracle.HostShard(K, rows, cols, t0=T0, dt=SEC, seed=4242)
        q2 = AggQuery(small, calls, 60 * SEC, T0, tmax, filter=flt).run()
        got, ref = q2.dense_host(), oracle.scan(hs.desc, q2.desc, threads=1)
        for k in range(len(calls)):
            rv = ref["cols"][k]["valid"].astype(bool)
            if not np.array_equal(got["cols"][k]["valid"].astype(bool), rv) or not np.array_equal(got["cols"][k]["values"].view(np.uint64)[rv], ref["cols"][k]["values"][rv]):
                raise VerifyError(f"mixed workload: call {k} differs from the oracle on the {K}-series slice")
        d = q.dense_host()
        verify = {"slice_series_bitwise_vs_oracle": K, "rows_counted_after_filter": int((d["cols"][0]["values"].astype(np.int64) * d["cols"][0]["valid"]).sum())}
        q2.close(); small.close()
    peak, peak_src = measured_peak()
    algo = st["page_bytes"] + st["dir_bytes"] + st["out_bytes"]
    k_ms = main_ms / a.steps
    line = {"metric": "decoded+aggregated rows/s", "value": info["n_rows"] * a.steps / (dev_ms / 1e3), "unit": "rows/s", "n_gpus": 1, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64+f64+u8", "data": "synthetic", "impl": "ours",
            "config": {"workload": f"configs[2]: {series} series x {rows} rows, int64 (Simple8b) + float64 (Gorilla G-lo) + bool columns, {a.nulls / 10:.0f}% nulls, "
                                   "count(i), sum(i), sum(f), count(b) WHERE f > 1000 GROUP BY time(1m), one tagset", "rows": int(info["n_rows"]),
                       "page_bytes": int(info["page_bytes"]), "compressed_bytes_per_row": info["page_bytes"] / max(1, info["n_rows"]),
                       "l2": "3 GB of pages per step: far larger than the 126 MB L2; no explicit flush"},
            "clocks": clocks, "roofline": {"bound": "hbm", "kernel": "k_fused_cols" if st["path"] == 5 else "k_fused_multi", "achieved": algo / (k_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                           "frac": algo / (k_ms / 1e3) / 1e9 / peak, "traffic": ncu_traffic(a) if st["path"] == 5 else None, "peak_source": peak_src, "algorithmic_bytes_per_launch": algo,
                                           "kernel_ms": k_ms, "note": "instruction-bound: three codecs decoded per row by one thread; bytes per row are ~3"},
            "e2e": None, "cpu_baseline": None, "verify": verify, "gpu_launches": launches, "path": st["path"]}
    print(json.dumps(line), flush=True)
    q.close(); sh.close()


def run_downsample(a):
    """configs[4] on one GPU (one of its 8 shards): 125 series x 10^6 float64 rows (1.25e8 rows), decode -> per-series
    min/max/sum/count/first/last per 5-minute window -> re-encode the six columns + time to TSSP pages with the device encoders
    (opengemini_b200/downsample.py: og_query_run with OG_GROUP_PER_SERIES, then og_encode_pages per output column).  One step = the
    whole read-aggregate-write pass, host wall clock around it with a device synchronize on both sides (the directory of the new
    shard is assembled on the host, so the step is not a pure device region).  Checked every run: the new shard is reopened and
    sum(count_) over it equals the source row count, min(min_) / max(max_) equal a direct query of the source."""
    import numpy as np
    import torch
    from opengemini_b200 import AggQuery, Shard
    from opengemini_b200 import _lib as L
    from opengemini_b200.downsample import downsample
    torch.cuda.set_device(0)
    Shard.init(0)
    series = a.series if a.series != 10_000 else 125
    rows = a.rows
    sh = Shard.synth(series, rows, [(L.TYPE_FLOAT, L.SYNTH_F_HI if a.dist == "hi" else L.SYNTH_F_LO, 0)], t0=T0, dt=SEC, seed=99)
    info = sh.info()
    tmax = T0 + (rows - 1) * SEC
    ivl = 300 * SEC
    for _ in range(max(a.warmup, 3)):
        out = downsample(sh, 0, ivl, T0, tmax)
    sampler = ClockSampler(0); sampler.start()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(a.steps):
        out = downsample(sh, 0, ivl, T0, tmax)
    torch.cuda.synchronize(); wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if a.dump_outputs:
        # the new shard as the pass hands it back: page bytes and their directory (window times relative to T0)
        arrays = {"pages": out["data"][:out["data_len"]].cpu().numpy(), "sids": out["sids"], "series_seg_begin": out["series_seg_begin"],
                  "seg_tmin": out["seg_tmin"] - T0, "seg_tmax": out["seg_tmax"] - T0,
                  "time_page_off": out["time_page_off"], "time_page_len": out["time_page_len"]}
        for name, _typ, po, pl in out["columns"]:
            arrays[f"{name}_page_off"], arrays[f"{name}_page_len"] = po, pl
        dump_outputs(a.dump_outputs, arrays)
    verify = None
    if not a.no_verify:
        host = out["data"].cpu().numpy()[:out["data_len"]].copy()
        ds = Shard.open(host, out["sids"], out["series_seg_begin"], out["seg_tmin"], out["seg_tmax"], out["columns"], out["time_page_off"], out["time_page_len"])
        # rows of the new shard carry their window start as time: the first one lies up to one interval before T0
        q1 = AggQuery(ds, [("min", 0), ("max", 1), ("sum", 3)], 0, T0 - ivl, tmax).run(); d1 = q1.dense_host()
        q0 = AggQuery(sh, [("min", 0), ("max", 0), ("count", 0)], 0, T0, tmax).run(); d0 = q0.dense_host()
        for k in range(3):
            if int(d1["cols"][k]["values"].view(np.uint64)[0]) != int(d0["cols"][k]["values"].view(np.uint64)[0]):
                raise VerifyError(f"downsample: aggregate {k} of the re-encoded shard differs from the source")
        verify = {"rows_counted_in_output": int(d1["cols"][2]["values"].view(np.int64)[0]), "output_rows": int(out["rows"]), "output_page_bytes": int(out["data_len"])}
        q1.close(); q0.close(); ds.close()
    line = {"metric": "decoded+aggregated rows/s", "value": info["n_rows"] * a.steps / wall, "unit": "rows/s", "n_gpus": 1, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": wall / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "ours",
            "config": {"workload": f"configs[4], one shard of eight: {series} series x {rows} float64 rows -> min/max/sum/count/first/last per series per 5 m -> re-encoded pages",
                       "rows": int(info["n_rows"]), "page_bytes_in": int(info["page_bytes"]), "timing": "host wall clock around the whole pass, device synchronised on both sides"},
            "clocks": clocks, "roofline": None, "e2e": None, "cpu_baseline": None, "verify": verify, "gpu_launches": None}
    print(json.dumps(line), flush=True)
    sh.close()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "mixed":
        run_mixed(args)
    elif args.workload == "downsample":
        run_downsample(args)
    else:
        run_ours(args)
