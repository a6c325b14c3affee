#!/usr/bin/env python
"""bench.py — shuffle rows/sec on the BASELINE.json workload.

Workload (config.workload = "cfg2"): 2^26 rows x 8 Int64 columns, col0 = uniform
i64 key, cols 1-7 = row_id*8+j, Hash([col0], 8) — BASELINE.json configs[1].
One "step" = one pass of the hot path over the whole table.

  value     rows/s with inputs resident in HBM (CUDA events on the library's stream)
  roofline  dominant kernel (k_scatter): algorithmic bytes (2*C*w per row) / its
            CUDA-event duration inside the timed region, vs MEASURED_PEAKS.json
  e2e       same metric through the C-ABI with HOST (pinned) buffers, H2D+D2H timed
  cpu_baseline  the oracle port of DataFusion's RepartitionExec on the host cores

`--impl reference` times the CPU path only (the oracle port, all host threads).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "shuffle rows/sec (64M rows, 8xi64, 8-way hash repartition)"
N_ROWS = 1 << 26
N_COLS = 8
WIDTH = 8
NUM_PARTITIONS = 8


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled (one `nvidia-smi -lms 100` process) while the GPU is
    under load: started before an untimed soak of the same step and stopped after the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.index = index
        self.samples = []
        self._p = None
        self._t = None

    def _run(self):
        for line in self._p.stdout:
            parts = [x.strip() for x in line.strip().split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def __enter__(self):
        try:
            self._p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                                        "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        except Exception:
            self._p = None
        return self

    def __exit__(self, *a):
        if self._p is not None:
            self._p.terminate()
            try:
                self._p.wait(timeout=5)
            except Exception:
                self._p.kill()
            self._t.join(timeout=5)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}

        def num(x):
            try:
                return float(x)
            except ValueError:
                return None

        sm = sorted(v for v in (num(s[0]) for s in self.samples) if v is not None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        pw = [v for v in (num(s[2]) for s in self.samples) if v is not None]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": num(self.samples[0][1]), "reasons": reasons,
                "samples": len(self.samples), "power_w_max": max(pw) if pw else None}


def bind_to_gpu_numa_node(index: int):
    """Pin this worker process to the CPU cores of its GPU's NUMA node BEFORE any pinned allocation, so that the
    page-locked staging buffers are node-local to the GPU's PCIe root (standard one-worker-per-GPU deployment).
    Returns (original affinity, description); a no-op when sysfs / nvidia-smi do not expose the topology."""
    try:
        orig = os.sched_getaffinity(0)
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if not bus:
            return None, "numa: unknown (no nvidia-smi)"
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None, "numa: single node"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= orig
        if not cpus:
            return None, f"numa: node {node} has no allowed cpus"
        os.sched_setaffinity(0, cpus)
        return orig, f"numa: bound to node {node} ({len(cpus)} cpus) of GPU {index}"
    except Exception as e:  # pragma: no cover - topology files missing
        return None, f"numa: not bound ({type(e).__name__})"


def nvlink_bytes(index: int):
    """(tx_bytes, rx_bytes) summed over the NVLink links of GPU `index`, from `nvidia-smi nvlink -gt d`; None if unavailable."""
    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(index)], capture_output=True, text=True, timeout=20).stdout
        tx = rx = 0
        seen = False
        for line in out.splitlines():
            line = line.strip()
            if "Data Tx:" in line or "Data Rx:" in line:
                val = line.split(":")[-1].strip().split()
                n = float(val[0]) * {"KiB": 1024, "MiB": 1 << 20, "GiB": 1 << 30, "B": 1}.get(val[1] if len(val) > 1 else "KiB", 1024)
                seen = True
                if "Tx" in line:
                    tx += n
                else:
                    rx += n
        return (tx, rx) if seen else None
    except Exception:
        return None


def soak(step, seconds: float, sync):
    """Untimed repetitions of the step so clocks/thermals are at steady state and the sampler sees load."""
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        for _ in range(20):
            step()
        sync()


def cpu_pool_arm(n_rows: int, steps: int, warmup: int, budget_s: float):
    """The reference's CPU path for this workload on the host cores: oracle port of RepartitionExec(Hash) +
    LimitedBatchCoalescer on a PERSISTENT worker pool with per-thread reusable buffers (oracle/df_oracle.c
    `orc_repartition_stream`; the reference's workers run tokio + mimalloc, benchmarks/cdk/bin/worker.rs:32).
    Thread-count sweep on a 2^24-row sample, then `steps` timed passes over the full table with the best count.
    Returns (rows_per_s, ms_per_step, steps_done, info)."""
    from oracle import oracle as orc
    from tests.util import cfg2_columns

    t_all = time.perf_counter()
    cores = os.cpu_count() or 1
    cols = cfg2_columns(n_rows, N_COLS)
    pool = orc.WorkerPool(cores)
    sample_rows = min(n_rows, 1 << 24)
    sample = [c[:sample_rows] for c in cols]
    cand = sorted({t for t in (1, 4, 8, 16, 32, 48, 64, 96, 128, 192, 256, cores) if t <= cores})
    sweep = {}
    for t in cand:
        pool.repartition(sample, [0], NUM_PARTITIONS, 8192, t)  # warm this thread count's buffers
        t0 = time.perf_counter()
        counts, _ = pool.repartition(sample, [0], NUM_PARTITIONS, 8192, t)
        sweep[t] = sample_rows / (time.perf_counter() - t0)
        assert int(counts.sum()) == sample_rows
    best_t = max(sweep, key=sweep.get)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        counts, batches = pool.repartition(cols, [0], NUM_PARTITIONS, 8192, best_t)
        dt = time.perf_counter() - t0
        assert int(counts.sum()) == n_rows
        if i >= warmup:
            times.append(dt)
        if time.perf_counter() - t_all > budget_s and times:
            break
    pool.close()
    ms = 1e3 * sum(times) / len(times)
    info = {"threads_used": best_t, "threads_swept": {str(k): round(v) for k, v in sweep.items()}, "one_thread_rows_per_s": round(sweep[min(sweep)]),
            "sweep_sample_rows": sample_rows, "rows_per_step": n_rows}
    return n_rows / (ms / 1e3), ms, len(times), info


CPU_WHAT = ("oracle port of DataFusion RepartitionExec(Hash) + LimitedBatchCoalescer (create_hashes -> index vectors -> take per "
            "(destination, column) -> coalesce to 8192-row batches), persistent thread pool, one input partition per thread, per-thread "
            "reusable buffers, consumers drop completed batches")


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path on the host cores.
    N = 1: local `RepartitionExec(Hash)` (BASELINE configs[1]: "vs CPU RepartitionExec") over the FULL 2^26-row table.
    N > 1: N producer tasks -> N consumer tasks: CPU repartition + Arrow Flight (IPC + LZ4, localhost gRPC)
           exchange — `oracle/flight_proxy.py`, the stand-in for impl_execute_task + WorkerConnectionPool.
    The real crate cannot be built here (no Rust toolchain), so both are the oracle port ("kind": "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    world = max(1, args.gpus)
    extra = {}
    if world == 1:
        v, ms, steps_done, info = cpu_pool_arm(args.rows, args.steps, args.warmup, 150.0)
        sample_rows = args.rows
        sample_txt = f"full {sample_rows}-row table per step; {CPU_WHAT}"
        extra.update(info)
        cores_used = info["threads_used"]
    else:
        import pyarrow as pa

        from oracle import oracle as orc
        from oracle.flight_proxy import FlightShuffleProxy
        from tests.util import cfg2_columns

        t_all = time.perf_counter()
        sample_rows = 1 << 23
        cols = cfg2_columns(sample_rows, N_COLS)
        # torchrun exports OMP_NUM_THREADS=1, which Arrow would take as its CPU pool size (IPC/LZ4 threads):
        # give the reference arm every host core, as the tokio runtime of the real workers would have
        pa.set_cpu_count(threads)
        pa.set_io_thread_count(max(8, min(64, threads)))
        total_parts = NUM_PARTITIONS if NUM_PARTITIONS % world == 0 else NUM_PARTITIONS * world
        P = total_parts // world
        names = [f"c{j}" for j in range(N_COLS)]
        prod = [[c[r * sample_rows // world:(r + 1) * sample_rows // world] for c in cols] for r in range(world)]
        tpp = max(1, threads // world)
        what = (f"{world} producer tasks -> {world} consumer tasks in one process: {CPU_WHAT} (Hash({total_parts}), all {threads} host threads) "
                f"+ pyarrow.flight localhost gRPC exchange, Arrow IPC with LZ4_FRAME (the reference default); charged max(repartition, exchange)")
        sample_txt = f"{sample_rows} rows (1/8 of the 2^26-row workload) per step; {what}"
        # producer half on the persistent pool (all producers' rows, all host threads)
        pool = orc.WorkerPool(threads)
        pool.repartition(cols, [0], total_parts, 8192, threads)
        t0 = time.perf_counter()
        pool.repartition(cols, [0], total_parts, 8192, threads)
        rep_s = time.perf_counter() - t0
        pool.close()
        px = FlightShuffleProxy(names, world, world, P, "lz4")
        vals, phases = [], []
        for i in range(args.warmup + args.steps):
            dt, rows, _ = px.run(prod, tpp)
            assert rows == sample_rows
            if i >= args.warmup:
                # charge the reference max(partition, exchange): its workers overlap the two phases
                vals.append(max(rep_s, px.last_phases[1]))
                phases.append((rep_s, px.last_phases[1]))
            if time.perf_counter() - t_all > 120 and len(vals) >= 1:
                break
        px.close()
        px = FlightShuffleProxy(names, world, world, P, None)  # uncompressed, for context
        px.run(prod, tpp)
        dt_nc, _, _ = px.run(prod, tpp)
        exch_nc = px.last_phases[1]
        px.close()
        extra["uncompressed_exchange_rows_per_s"] = sample_rows / exch_nc
        extra["phase_ms"] = {"repartition": 1e3 * rep_s, "flight_exchange": 1e3 * sum(p[1] for p in phases) / len(phases),
                             "charged": "max(repartition, exchange) — assumes the reference overlaps the two phases perfectly"}
        ms = 1e3 * sum(vals) / len(vals)
        v = sample_rows / (ms / 1e3)
        steps_done = len(vals)
        cores_used = threads
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "rows/s", "n_gpus": args.gpus, "steps": steps_done,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": "cfg2: 2^26 rows x 8 Int64, Hash([col0], 8), batch 8192" + ("" if world == 1 else "; bounded sample"),
                   "rows_per_step": sample_rows},
        "cpu_baseline": dict({"value": v, "unit": "rows/s", "cores": cores_used, "host_cores": threads, "kind": "port", "sample": sample_txt}, **extra),
        "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def measure_pcie(torch, mib: int = 256, reps: int = 6):
    """Measured PCIe copy rates of this box (pinned host memory <-> HBM, CUDA events): each direction alone and both at
    once on two streams — the ceiling of the host-to-host (`e2e`) number, which moves every byte once in each direction."""
    nbytes = mib << 20
    h_in, h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory(), torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_a, d_b = torch.empty(nbytes, dtype=torch.uint8, device="cuda"), torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def run(h2d: bool, d2h: bool) -> float:
        torch.cuda.synchronize()
        start = torch.cuda.Event(enable_timing=True)
        start.record()
        ends = []
        for on, st, dst, src in ((h2d, s1, d_a, h_in), (d2h, s2, h_out, d_b)):
            if not on:
                continue
            st.wait_event(start)
            with torch.cuda.stream(st):
                for _ in range(reps):
                    dst.copy_(src, non_blocking=True)
                e = torch.cuda.Event(enable_timing=True)
                e.record(st)
                ends.append(e)
        torch.cuda.synchronize()
        return max(start.elapsed_time(e) for e in ends) / 1e3

    run(True, True)
    total = nbytes * reps / 1e9
    out = {"h2d_gbs": total / run(True, False), "d2h_gbs": total / run(False, True), "duplex_gbs_per_direction": total / run(True, True),
           "how": f"{reps} x {mib} MiB pinned copies per direction, CUDA events"}
    del h_in, h_out, d_a, d_b
    return out


def run_e2e(ctx, dfd, n, args):
    """Same metric through the reference-facing operator (RepartitionExec over the C-ABI)
    with HOST buffers: pinned Arrow record batches in, per-destination Arrow batches out,
    H2D and D2H copies inside the timed region (wall clock around push..finish..drain)."""
    import pyarrow as pa

    names = [f"c{j}" for j in range(N_COLS)]
    pt = dfd.PinnedTable(ctx, n, [np.int64] * N_COLS)
    rng = np.random.Generator(np.random.PCG64(42))
    step = 1 << 22
    for lo in range(0, n, step):
        hi = min(lo + step, n)
        pt.columns[0][lo:hi] = rng.integers(-(2**63), 2**63 - 1, hi - lo, dtype=np.int64, endpoint=True)
        rid = np.arange(lo, hi, dtype=np.int64)
        for j in range(1, N_COLS):
            pt.columns[j][lo:hi] = rid * 8 + j
    batches = pt.record_batches(names, args.e2e_batch_rows)
    schema = batches[0].schema
    times = []
    st = None
    for it in range(2 + args.steps):
        ex = dfd.RepartitionExec(ctx, schema, dfd.Partitioning.Hash([0], NUM_PARTITIONS), chunk_rows=args.e2e_chunk_rows,
                                 pipeline_depth=3, pinned_pool_chunks=args.e2e_pool_chunks)
        readers = [ex.execute(p) for p in range(NUM_PARTITIONS)]
        counts = [0] * NUM_PARTITIONS

        def consume(p):  # one consumer per destination stream, like the reference's per-partition pollers
            for rb in readers[p]:
                counts[p] += rb.num_rows

        consumers = [threading.Thread(target=consume, args=(p,)) for p in range(NUM_PARTITIONS)]
        t0 = time.perf_counter()
        for t in consumers:
            t.start()
        for b in batches:
            ex.push_batch(b)
        ex.finish()
        for t in consumers:
            t.join()
        dt = time.perf_counter() - t0
        rows_out = sum(counts)
        assert rows_out == n, (rows_out, n)
        st = ex.stats()
        del readers
        ex.close()
        if it >= 2:
            times.append(dt)
    best = sum(times) / len(times)
    pt.close()
    import torch

    try:
        pcie = measure_pcie(torch)
        pcie_frac = (int(st["bytes_h2d"]) / best / 1e9) / pcie["duplex_gbs_per_direction"]
    except Exception as e:  # (e.g. no pinned memory left on a loaded host: the e2e number itself does not depend on it)
        pcie, pcie_frac = {"error": str(e)[:200]}, None
    return {"value": n / best, "unit": "rows/s", "h2d_bytes_per_step": int(st["bytes_h2d"]), "d2h_bytes_per_step": int(st["bytes_d2h"]),
            "ms_per_step": best * 1e3, "steps": len(times), "batch_rows": args.e2e_batch_rows, "chunk_rows": args.e2e_chunk_rows,
            "api": "RepartitionExec.push_batch/finish/execute(partition) over dfd_repartition_exec_* (Arrow C Data / C Stream)",
            # the last operator of the loop: pinned output chunks it held / pinned itself / took over from the context's cache,
            # and where the producer thread's time went
            "operator": {"pinned_chunks": int(st["pinned_chunks"]), "pinned_chunks_allocated": int(st["pinned_chunks_allocated"]),
                         "pinned_chunks_reused": int(st["pinned_chunks_reused"]), "push_ms": st["ns_push"] / 1e6,
                         "wait_d2h_ms": st["ns_wait_d2h"] / 1e6, "wait_pool_ms": st["ns_wait_pool"] / 1e6},
            "pcie": pcie, "frac_of_pcie_duplex": pcie_frac}


DUMP_SAMPLE_ROWS = 1 << 18  # rows sampled by --dump-outputs: 17 float64 arrays of 2 MiB (36 MB) stay under 64 MB


def dump_outputs(out_dir, torch, outs, starts, counts):
    """Write what the last timed step handed its caller, so that two builds can be compared output for output:
    `partition_counts` (rows per destination) and, for a fixed seeded sample of positions in destination order
    (`sample_positions`; destination p is rows [starts[p], starts[p] + counts[p]) of every output column), each
    int64 output column as `col<c>_hi` / `col<c>_lo`, its signed high and unsigned low 32 bits in float64, which
    round-trip exactly.  Every array is float64."""
    os.makedirs(out_dir, exist_ok=True)
    n = int(counts.sum())
    rng = np.random.Generator(np.random.PCG64(20261017))
    pos = np.arange(n) if n <= DUMP_SAMPLE_ROWS else np.sort(rng.choice(n, DUMP_SAMPLE_ROWS, replace=False))
    first = np.concatenate([[0], np.cumsum(counts)])
    dest = np.searchsorted(first, pos, side="right") - 1
    idx = torch.from_numpy(starts[dest] + (pos - first[dest])).to(outs[0].device)
    arrays = {"partition_counts": counts, "sample_positions": pos}
    for c, col in enumerate(outs):
        v = col.index_select(0, idx).cpu().numpy()
        arrays[f"col{c}_hi"], arrays[f"col{c}_lo"] = v >> 32, v & 0xFFFFFFFF
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


TRAFFIC_ONEPASS = 8.564484e9  # dram__bytes_read.sum + dram__bytes_write.sum of one k_scatter_onepass launch at cfg-2 (profiles/r02c_ncu_summary.md)
NVLINK_PEAK_GBS = 770.0  # measured peer copy per direction per GPU on this pool (B200_PROFILING.md; nominal 900)


def multi_gpu_parity(args, torch, dist, dfd, nv, ctx, ex, world, rank, P, total_parts):
    """Bit-parity of the multi-GPU shuffle against the single-node CPU oracle, run by EVERY rank before the timed
    region (the reference's correctness bar is distributed == single node, tests/tpch_correctness_test.rs:137-146).
    A seeded cfg-2 table of `parity_rows` rows is split into contiguous producer ranges; every consumer compares each
    of its partitions — per producer segment, values AND order — with the oracle's rows for that (destination, producer).
    Returns the number of mismatching segments summed over ranks (0 == parity)."""
    import uuid

    from oracle import oracle as orc
    from tests.util import cfg2_columns

    n_chk = args.parity_rows
    cols = cfg2_columns(n_chk, N_COLS, seed=1234)
    lo, hi = rank * n_chk // world, (rank + 1) * n_chk // world
    ins = [torch.from_numpy(c[lo:hi].copy()).cuda() for c in cols]
    torch.cuda.synchronize()
    in_cols = [dfd.DeviceColumn.from_torch(t) for t in ins]
    dest = orc.partition_ids([cols[0]], n_chk, total_parts)
    node = dfd.NetworkShuffleExec.try_new(dfd.Partitioning.Hash([0], P), uuid.uuid4(), 99, world, world)
    bad = 0

    def fetch(col, a, cnt):
        got = np.empty(cnt, dtype=np.int64)
        if cnt:
            nv.check(nv.lib().dfd_memcpy_d2h(ctx.handle, got.ctypes.data, col.values + a * 8, cnt * 8))
        return got

    if args.exchange == "onepass":
        node.shuffle_onepass(ex, in_cols, hi - lo)
        node.shuffle_onepass(ex, in_cols, hi - lo)  # twice: window reuse is ordered by the ready/done flags
        outs, seg_starts, seg_counts = node.collect(ex)
        segs = lambda q, r: (int(seg_starts[q, r]), int(seg_counts[q, r]))
    else:
        cap = int((hi - lo) * 1.5) + 4096
        mode = nv.EXCHANGE_FUSED if args.exchange == "fused" else nv.EXCHANGE_NCCL
        outs_t = [torch.empty(cap, dtype=torch.int64, device="cuda") for _ in range(N_COLS)] if mode == nv.EXCHANGE_NCCL else None
        out_cols = [dfd.DeviceColumn.from_torch(t) for t in outs_t] if outs_t else None
        outs, starts = node.shuffle(ex, in_cols, hi - lo, mode, out_cols, cap)
        per = {}
        for q in range(P):
            run = int(starts[q])
            for r in range(world):
                cnt = int(np.count_nonzero(dest[r * n_chk // world:(r + 1) * n_chk // world] == rank * P + q))
                per[(q, r)] = (run, cnt)
                run += cnt
            if run != int(starts[q + 1]):
                bad += 1
        segs = lambda q, r: per[(q, r)]
    for q in range(P):
        g = rank * P + q
        for r in range(world):
            rlo, rhi = r * n_chk // world, (r + 1) * n_chk // world
            want = np.nonzero(dest[rlo:rhi] == g)[0] + rlo
            a, cnt = segs(q, r)
            if cnt != len(want):
                bad += 1
                continue
            for c in range(N_COLS):
                if not np.array_equal(fetch(outs[c], a, cnt), cols[c][want]):
                    bad += 1
    t = torch.tensor([bad], dtype=torch.int64, device="cuda")
    dist.all_reduce(t)
    return int(t.item())


def run_multi_gpu(args, torch, dfd, world):
    """N workers = N GPUs of one NVSwitch box, one rank per GPU.  Strong scaling: the 2^26-row
    table is split into `world` contiguous row ranges (producer tasks); N = 8 global partitions,
    P = 8/world per consumer task.  One step = one collective shuffle:
      onepass : k_xchg_signal_ready -> k_scatter_onepass<PEER> (hash once, look-back, peer stores) -> k_xchg_publish_wait
      fused   : hist + count all-gather + two-pass peer-store scatter + NCCL barrier
      nccl    : local partition + grouped ncclSend/ncclRecv
    Timed with CUDA events on the library stream, max over ranks.  Before the timed region every rank checks
    bit-parity against the CPU oracle on a seeded slice (parity_checked / parity_rows in the JSON line); a mismatch
    fails the run."""
    import uuid

    import torch.distributed as dist

    from datafusion_distributed_b200 import _native as nv

    rank = int(os.environ["RANK"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_total = args.rows
    total_parts = NUM_PARTITIONS if NUM_PARTITIONS % world == 0 else NUM_PARTITIONS * world
    P = total_parts // world
    lo, hi = rank * n_total // world, (rank + 1) * n_total // world
    n = hi - lo
    g = torch.Generator(device="cuda").manual_seed(42 + rank)
    key = torch.randint(-(2**63), 2**63 - 1, (n,), dtype=torch.int64, device="cuda", generator=g)
    rid = torch.arange(lo, hi, dtype=torch.int64, device="cuda")
    ins = [key] + [rid * 8 + j for j in range(1, N_COLS)]
    del rid
    cap = int(n * 1.25) + 4096
    torch.cuda.synchronize()
    uid = [dfd.nccl_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    ctx = dfd.WorkerContext(local_rank)
    ex = dfd.ShuffleExchange(ctx, rank, world, uid[0])
    mode = {"onepass": None, "fused": nv.EXCHANGE_FUSED, "nccl": nv.EXCHANGE_NCCL}[args.exchange]
    ex.setup_window(cap * N_COLS * WIDTH)
    outs_t = [torch.empty(cap, dtype=torch.int64, device="cuda") for _ in range(N_COLS)] if mode == nv.EXCHANGE_NCCL else None
    torch.cuda.synchronize()
    in_cols = [dfd.DeviceColumn.from_torch(t) for t in ins]
    out_cols = [dfd.DeviceColumn.from_torch(t) for t in outs_t] if outs_t else None
    node = dfd.NetworkShuffleExec.try_new(dfd.Partitioning.Hash([0], P), uuid.uuid4(), 1, world, world)

    parity_bad = multi_gpu_parity(args, torch, dist, dfd, nv, ctx, ex, world, rank, P, total_parts)
    if parity_bad:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "n_gpus": world, "parity_checked": False, "parity_mismatching_segments": parity_bad,
                              "error": "multi-GPU shuffle differs from the CPU oracle"}))
        ex.close()
        dist.destroy_process_group()
        sys.exit(3)

    def step():
        if mode is None:
            node.shuffle_onepass(ex, in_cols, n)
            return node.collect(ex)
        return node.shuffle(ex, in_cols, n, mode, out_cols, cap)

    def timed_steps(k):
        """K back-to-back shuffles; the fused transports are enqueued asynchronously (like the 1-GPU path's launches)
        and synchronised once at the end, the NCCL transport needs the host count exchange every step."""
        if mode is None:
            for _ in range(k):
                node.shuffle_onepass(ex, in_cols, n)
            _, _, seg_counts = node.collect(ex)
            return int(seg_counts.sum())
        if mode == nv.EXCHANGE_FUSED:
            for _ in range(k):
                node.shuffle_async(ex, in_cols, n)
            return int(node.wait(ex)[1][-1])
        r = None
        for _ in range(k):
            r = step()
        return int(r[1][-1])

    with ClockSampler(local_rank) as clocks:  # started before warm-up: nvidia-smi needs ~1 s to deliver its first sample
        for _ in range(max(args.warmup, 3)):
            step()
        # untimed soak (collective: the same count on every rank), sized for >= ~2 s under load
        if not args.no_soak:
            timed_steps(2500 if mode != nv.EXCHANGE_NCCL else 300)
        ctx.reset_metrics()
        dist.barrier()
        torch.cuda.synchronize()
        ctx.synchronize()
        ctx.timer_start()
        got_rows = timed_steps(args.steps)
        ms_local = ctx.timer_stop()
    torch.cuda.synchronize()
    dist.barrier()
    t = torch.tensor([ms_local], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = t.item() / args.steps
    recv_rows = torch.tensor([got_rows], dtype=torch.int64, device="cuda")
    dist.all_reduce(recv_rows)
    assert recv_rows.item() == n_total, (recv_rows.item(), n_total)
    launches = torch.tensor([int(ctx.metrics()["kernel_launches"])], dtype=torch.int64, device="cuda")
    dist.all_reduce(launches)
    fallbacks = int(nv.lib().dfd_exchange_onepass_fallbacks(ex._h))
    # phase split of the step (separate, untimed loop with per-phase CUDA events) + NVLink byte counters around it
    phases = None
    nvl = None
    if mode is None:
        import ctypes as C

        nv0 = nvlink_bytes(local_rank)
        ctx.set_profiling(True)
        k_prof = 50
        timed_steps(k_prof)
        out3, cnt = (C.c_double * 3)(), C.c_uint64()
        nv.check(nv.lib().dfd_exchange_phase_ms(ex._h, out3, C.byref(cnt)))
        ctx.set_profiling(False)
        nv1 = nvlink_bytes(local_rank)
        ph = torch.tensor(list(out3), dtype=torch.float64, device="cuda")
        ph_max = ph.clone()
        dist.all_reduce(ph_max, op=dist.ReduceOp.MAX)
        phases = {"signal_ready_ms": ph_max[0].item(), "scatter_ms": ph_max[1].item(), "publish_wait_ms": ph_max[2].item(),
                  "rank0": {"signal_ready_ms": out3[0], "scatter_ms": out3[1], "publish_wait_ms": out3[2]},
                  "how": f"CUDA events around the three stream phases of {int(cnt.value)} untimed shuffles; max over ranks"}
        if nv0 and nv1:
            nvl = {"tx_bytes_per_shuffle": (nv1[0] - nv0[0]) / k_prof, "rx_bytes_per_shuffle": (nv1[1] - nv0[1]) / k_prof,
                   "source": "nvidia-smi nvlink -gt d (sum over links of this GPU), rank 0, around the untimed phase-timing loop"}

    # e2e: host (pinned) rows in, host rows out, per worker, through dfd_shuffle_host: chunked
    # H2D | fused shuffle | D2H pipeline (every chunk is one collective), wall clock, max over ranks
    e2e = None
    if not args.no_e2e:
        pt_in = dfd.PinnedTable(ctx, n, [np.int64] * N_COLS)
        pt_out = dfd.PinnedTable(ctx, cap, [np.int64] * N_COLS)
        for j in range(N_COLS):
            nv.check(nv.lib().dfd_memcpy_d2h(ctx.handle, pt_in.columns[j].ctypes.data, ins[j].data_ptr(), n * WIDTH))
        h_in = [dfd.DeviceColumn(nv.COL_FIXED, WIDTH, a.ctypes.data, length=n) for a in pt_in.columns]
        h_out = [dfd.DeviceColumn(nv.COL_FIXED, WIDTH, a.ctypes.data, length=cap) for a in pt_out.columns]
        n_chunks = max(2, min(16, n // (1 << 20)))
        e2e_times = []
        got = 0
        for it in range(2 + args.steps):
            dist.barrier()
            t0 = time.perf_counter()
            cps = node.shuffle_host(ex, h_in, n, n_chunks, h_out, cap)
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            got = int(cps[-1, -1])
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            if it >= 2:
                e2e_times.append(dt.item())
        e2e_s = sum(e2e_times) / len(e2e_times)
        tot = torch.tensor([n * N_COLS * WIDTH, got * N_COLS * WIDTH, got], dtype=torch.int64, device="cuda")
        dist.all_reduce(tot)
        assert tot[2].item() == n_total
        e2e = {"value": n_total / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": int(tot[0].item()), "d2h_bytes_per_step": int(tot[1].item()),
               "ms_per_step": e2e_s * 1e3, "steps": len(e2e_times), "chunks_per_worker": n_chunks,
               "api": "per worker: NetworkShuffleExec.shuffle_host -> dfd_shuffle_host (pinned host columns in/out; chunked "
                      "H2D | fused shuffle | D2H pipeline); wall clock, max over ranks"}
        pt_in.close()
        pt_out.close()
    if rank == 0:
        alg = N_COLS * WIDTH * n * (world - 1) / world  # bytes each GPU must push through NVLink per direction
        achieved = alg / (ms_per_step / 1e3) / 1e9
        line = {
            "metric": METRIC, "value": n_total / (ms_per_step / 1e3), "unit": "rows/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": f"cfg2: 2^26 rows x 8 Int64 split over {world} producer tasks, Hash([col0], {total_parts}), "
                                   f"{P} partitions per consumer task, device-resident", "rows": n_total, "columns": N_COLS,
                       "num_partitions": total_parts, "exchange": args.exchange, "host": args.numa_note,
                       "l2": f"per-GPU inputs+window ({2 * n * N_COLS * WIDTH >> 20} MiB) > L2, no flush"},
            "parity_checked": True, "parity_rows": args.parity_rows,
            "parity": "every rank compared each (partition, producer) segment — values and order — with the single-node CPU oracle before the timed region",
            "onepass_fallbacks": fallbacks,
            "roofline": {"bound": "nvlink", "kernel": {"onepass": "k_scatter_onepass<PEER> (hash once -> look-back -> peer stores; flags over peer memory)",
                                                        "fused": "k_scatter<PEER> (two-pass; ncclAllGather(counts) + ncclAllReduce barrier)",
                                                        "nccl": "ncclSend/Recv"}[args.exchange],
                         "achieved": achieved, "peak": NVLINK_PEAK_GBS, "unit": "GB/s", "frac": achieved / NVLINK_PEAK_GBS,
                         "peak_source": "measured peer copy per direction (B200_PROFILING.md); nominal 900",
                         "traffic": (nvl["tx_bytes_per_shuffle"] if nvl else None), "traffic_unit": "NVLink Tx bytes per shuffle (rank 0)",
                         "nvlink_counters": nvl, "phases": phases,
                         "algorithmic_bytes_per_gpu_per_direction": alg},
            "gpu_launches": int(launches.item()), "clocks": clocks.summary(), "e2e": e2e,
        }
        print(json.dumps(line))
    ex.close()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=N_ROWS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-soak", action="store_true", help="skip the untimed clock soak (use under ncu)")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the worker to its GPU's NUMA node")
    ap.add_argument("--e2e-batch-rows", type=int, default=1 << 20)
    ap.add_argument("--e2e-chunk-rows", type=int, default=1 << 20)
    ap.add_argument("--e2e-pool-chunks", type=int, default=6, help="pinned output chunks the operator pre-allocates (the pool grows on demand)")
    ap.add_argument("--exchange", default="onepass", choices=["onepass", "fused", "nccl"],
                    help="multi-GPU transport: single-pass fused (peer stores + peer-memory flags), two-pass fused, or NCCL send/recv")
    ap.add_argument("--parity-rows", type=int, default=1 << 21, help="rows of the multi-GPU bit-parity check run before the timed region")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5", "agg", "fixture"],
                    help="cfg2 = the BASELINE.json headline (default; what the driver runs); cfg3/4/5 = the other configs (bench_workloads.py)")
    ap.add_argument("--kernel", default="onepass", choices=["onepass", "twopass"],
                    help="1-GPU partition path: single-pass k_scatter<ONEPASS> (regions) or K1/K1b/K2 (dense)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of the last step's "
                    "outputs as DIR/<name>.npy (float64; cfg2 on one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "cfg2" or args.gpus != 1):
        ap.error("--dump-outputs covers the cfg2 workload on one GPU")
    if args.impl == "reference":
        if args.workload == "cfg4":
            import bench_workloads

            return bench_workloads.run_reference_cfg4(args)
        return run_reference(args)

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    orig_affinity, numa_note = (None, "numa: binding disabled") if args.no_numa_bind else bind_to_gpu_numa_node(local_rank)
    args.numa_note = numa_note
    args.orig_affinity = orig_affinity

    import torch

    import datafusion_distributed_b200 as dfd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload != "cfg2":
        import bench_workloads

        return bench_workloads.run(args, torch, dfd, world)
    if world > 1:
        return run_multi_gpu(args, torch, dfd, world)
    if args.gpus != 1:
        raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    dev = 0
    torch.cuda.set_device(dev)
    n = args.rows
    g = torch.Generator(device="cuda").manual_seed(42)
    key = torch.randint(-(2**63), 2**63 - 1, (n,), dtype=torch.int64, device="cuda", generator=g)
    rid = torch.arange(n, dtype=torch.int64, device="cuda")
    ins = [key] + [rid * 8 + j for j in range(1, N_COLS)]
    del rid
    ctx = dfd.WorkerContext(dev)
    part = dfd.HashPartitioner(ctx, dfd.Partitioning.Hash([0], NUM_PARTITIONS))
    onepass = args.kernel == "onepass"
    region_rows = part.default_region_rows(n) if onepass else 0  # fair share + 25 % per destination
    outs = [torch.empty(NUM_PARTITIONS * region_rows if onepass else n, dtype=torch.int64, device="cuda") for _ in ins]
    torch.cuda.synchronize()
    in_cols = [dfd.DeviceColumn.from_torch(t) for t in ins]
    out_cols = [dfd.DeviceColumn.from_torch(t) for t in outs]

    def one_step():
        if onepass:
            part.partition_onepass(in_cols, n, region_rows, out_cols, sync=False)
        else:
            part.partition(in_cols, n, out_cols, sync=False)

    for _ in range(max(args.warmup, 3)):
        one_step()
    ctx.synchronize()
    ctx.reset_metrics()
    ctx.set_profiling(True)
    # inputs (4 GiB) + outputs (4 GiB) are far larger than the 126 MB L2: no flush needed between steps
    with ClockSampler(dev) as clocks:
        if not args.no_soak:
            soak(one_step, 1.0, ctx.synchronize)
        ctx.reset_metrics()
        ctx.timer_start()
        for _ in range(args.steps):
            one_step()
        ms_total = ctx.timer_stop()
    m = ctx.metrics()
    if onepass:
        starts, counts = part.collect()
        assert int(counts.sum()) == n and ctx.metrics()["onepass_reruns"] == 0, "a destination region overflowed inside the timed loop"
    ctx.set_profiling(False)
    if args.dump_outputs:
        if not onepass:  # dense layout: destination p is rows [part_starts[p], part_starts[p + 1])
            from datafusion_distributed_b200 import _native as nv

            bounds = np.empty(NUM_PARTITIONS + 1, dtype=np.int64)
            nv.check(nv.lib().dfd_memcpy_d2h(ctx.handle, bounds.ctypes.data, part.part_starts_device_ptr(), bounds.nbytes))
            starts, counts = bounds[:-1], np.diff(bounds)
        dump_outputs(args.dump_outputs, torch, outs, starts, counts)
    ms_per_step = ms_total / args.steps
    value = n / (ms_per_step / 1e3)

    peak, peak_src = measured_peaks()
    alg_bytes = 2.0 * N_COLS * WIDTH * n
    scatter_ms = m["scatter_ms"] / max(m["scatter_launches"], 1)
    achieved = alg_bytes / (scatter_ms / 1e3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": "cfg2: 2^26 rows x 8 Int64, Hash([col0], 8), device-resident table", "rows": n,
                   "columns": N_COLS, "num_partitions": NUM_PARTITIONS, "l2": "inputs+outputs (8 GiB) >> L2, no flush",
                   "kernel_path": ("single pass: k_scatter_onepass (TMA-fed ring, hash once, decoupled look-back, per-destination regions of "
                                   f"{region_rows} rows)") if onepass else "two pass: k_tile_hist -> k_scan_tiles -> k_scatter (dense)"},
        "roofline": {"bound": "hbm", "kernel": "k_scatter_onepass" if onepass else "k_scatter", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "peak_source": peak_src,
                     # dram__bytes_read.sum + dram__bytes_write.sum of one k_scatter launch at this exact workload,
                     # from the committed `ncu --set full` capture profiles/r01c_ncu_summary.md (8.59 GB algorithmic)
                     "traffic": (TRAFFIC_ONEPASS if onepass else 8.576116e9) if n == N_ROWS else None, "traffic_unit": "bytes/launch",
                     "traffic_source": "profiles/r02c_ncu_summary.md" if onepass else "profiles/r01c_ncu_summary.md",
                     "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": scatter_ms,
                     "hist_ms": m["hist_ms"] / max(m["calls"], 1), "scan_ms": m["scan_ms"] / max(m["calls"], 1)},
        "gpu_launches": int(m["kernel_launches"]),
        "clocks": clocks.summary(),
        "e2e": None,
    }
    if not args.no_e2e:
        line["e2e"] = run_e2e(ctx, dfd, n, args)
        line["gpu_launches"] = int(ctx.metrics()["kernel_launches"])
    line["config"]["host"] = args.numa_note
    if not args.no_cpu_baseline:
        if args.orig_affinity:
            os.sched_setaffinity(0, args.orig_affinity)  # the CPU baseline uses every host core
        v, ms_cpu, steps_cpu, info = cpu_pool_arm(n, 3, 1, 25.0)
        line["cpu_baseline"] = dict({"value": v, "unit": "rows/s", "cores": info["threads_used"], "host_cores": os.cpu_count() or 1, "kind": "port",
                                     "sample": f"full {n}-row table, mean of {steps_cpu} passes after 1 warm-up; {CPU_WHAT}"}, **info)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
