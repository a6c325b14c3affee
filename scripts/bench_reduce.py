"""bench_reduce.py — the device-side PartialReduce (dfd_partial_reduce_device) timed alone.

Each workload is generated from a fixed seed, partitioned by a destination column on the host (rows sorted by destination,
part_starts uploaded) and kept on the device; only the reduce call is inside the timed region, bracketed by the context's
CUDA-event stopwatch (dfd_timer_start / dfd_timer_stop) one call at a time.  The call ends with its own stream
synchronisation, so a timing covers the whole call, including its one host round trip for the group counts.

  int           4M rows, 65 536 Int64 groups, 8 partitions, SUM / COUNT / MIN / MAX over Int64 and a Decimal128 SUM:
                fixed-width, non-null columns only (the path that existed before nullable and string keys)
  raintoday     2^24 rows, one nullable Utf8 key in {"Yes", "No", NULL}, COUNT, 8 partitions: three groups per
                partition, so the atomics on a few output rows dominate
  searchphrase  2^24 rows, a zipf-distributed Utf8 key over 2^18 phrases with 30 % empty strings and 2 % NULLs, COUNT
                plus a nullable SUM, 8 partitions
  q1            TPC-H q1's partial-aggregate shape (cfg-3): 24 rows, (l_returnflag, l_linestatus) Utf8 keys, 10 nullable
                states (4 x Decimal128 SUM, 4 x Int64 SUM, Float64 MIN / MAX), 3 partitions; latency bound, reported in us

Prints one JSON line per workload with the median, min, max and 10th / 90th percentiles in ms, and the GPU's name and
power limit (read-only nvidia-smi query).  Needs a GPU: without one it exits with an error and measures nothing."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = ["int", "raintoday", "searchphrase", "q1"]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30, check=True).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001 (reported, not fatal: the timing itself comes from CUDA events)
        return f"unknown ({e.__class__.__name__})", "unknown"


def by_destination(dest, N):
    order = np.argsort(dest, kind="stable")
    starts = np.zeros(N + 1, dtype=np.int64)
    starts[1:] = np.cumsum(np.bincount(dest, minlength=N))
    return order, starts


def strings(ids, vocab):
    """(offsets int32, bytes) of vocab[ids] without a Python loop over the rows."""
    lens = np.array([len(v) for v in vocab], np.int64)
    offs = np.r_[0, np.cumsum(lens[ids])].astype(np.int32)
    blob = np.frombuffer(b"".join(vocab), np.uint8)
    vstart = np.r_[0, np.cumsum(lens)[:-1]]
    data = blob[np.repeat(vstart[ids] - offs[:-1], lens[ids]) + np.arange(int(offs[-1]))]
    return offs, data


def bits(valid):
    b = np.packbits(valid.astype(np.uint8), bitorder="little")
    return np.concatenate([b, np.zeros((-len(b)) % 8 + 8, np.uint8)])


def make(workload, rng):
    """-> (columns as dicts {kind, width, values, offsets, validity}, key indices, ops, dest, N)."""
    from datafusion_distributed_b200 import _native as nv

    fixed = lambda a, valid=None: {"kind": nv.COL_FIXED, "width": a.dtype.itemsize * (a.shape[1] if a.ndim == 2 else 1),  # noqa: E731
                                   "values": a, "validity": None if valid is None else bits(valid)}
    if workload == "int":
        n, G, N = 4 << 20, 1 << 16, 8
        g = rng.integers(0, G, n)
        key = (g.astype(np.uint64) * np.uint64(0x9E37_79B9_7F4A_7C15)).view(np.int64)
        dec = np.stack([rng.integers(0, 1 << 62, n, dtype=np.uint64), rng.integers(0, 4, n, dtype=np.uint64)], axis=1)
        cols = [fixed(key), fixed(rng.integers(-(1 << 40), 1 << 40, n)), fixed(np.ones(n, np.int64)),
                fixed(rng.integers(-(1 << 62), 1 << 62, n)), fixed(rng.integers(-(1 << 62), 1 << 62, n)), fixed(dec)]
        ops = [-1, nv.AGG_SUM_I64, nv.AGG_SUM_I64, nv.AGG_MIN_I64, nv.AGG_MAX_I64, nv.AGG_SUM_I128]
        return cols, [0], ops, g % N, N
    if workload in ("raintoday", "searchphrase"):
        n, N = 1 << 24, 8
        if workload == "raintoday":
            vocab = [b"Yes", b"No"]
            ids = rng.integers(0, 2, n)
            valid = rng.random(n) >= 0.1
        else:
            vocab = [b""] + [b"search phrase %d" % i + b" words" * (i % 11) for i in range(1, 1 << 18)]
            ids = (rng.zipf(1.1, n) - 1) % len(vocab)
            ids[rng.random(n) < 0.3] = 0
            valid = rng.random(n) >= 0.02
        offs, data = strings(ids, vocab)
        key = {"kind": nv.COL_UTF8, "width": 0, "values": data, "offsets": offs, "validity": bits(valid)}
        cols = [key, fixed(np.ones(n, np.int64))]
        ops = [-1, nv.AGG_SUM_I64]
        if workload == "searchphrase":
            cols.append(fixed(rng.integers(0, 1 << 20, n), rng.random(n) < 0.7))
            ops.append(nv.AGG_SUM_I64)
        gid = np.where(valid, ids, -1)
        return cols, [0], ops, (gid * 2_654_435_761) % N, N
    # q1
    groups = [(b"A", b"F"), (b"N", b"F"), (b"N", b"O"), (b"R", b"F")] * 6
    n, N = len(groups), 3
    cols = []
    for j in range(2):
        vocab = sorted({g[j] for g in groups})
        offs, data = strings(np.array([vocab.index(g[j]) for g in groups]), vocab)
        cols.append({"kind": nv.COL_UTF8, "width": 0, "values": data, "offsets": offs, "validity": None})
    ops = [-1, -1]
    for j in range(10):
        valid = rng.random(n) < 0.8
        if j < 4:
            cols.append(fixed(np.stack([rng.integers(0, 1 << 50, n, dtype=np.uint64), np.zeros(n, np.uint64)], axis=1), valid))
            ops.append(nv.AGG_SUM_I128)
        elif j < 8:
            cols.append(fixed(rng.integers(0, 1 << 40, n), valid))
            ops.append(nv.AGG_SUM_I64)
        else:
            cols.append(fixed(rng.standard_normal(n), valid))
            ops.append(nv.AGG_MIN_F64 if j == 8 else nv.AGG_MAX_F64)
    dest = np.arange(n) % N  # each partition holds every group of two input partitions
    return cols, [0, 1], ops, dest, N


def run(workload, iters, warmup):
    import torch

    import datafusion_distributed_b200 as dfd
    from datafusion_distributed_b200 import _native as nv

    ctx = dfd.WorkerContext(0)
    rng = np.random.Generator(np.random.PCG64(2024))
    cols, keys, ops, dest, N = make(workload, rng)
    order, starts = by_destination(np.asarray(dest), N)
    n = len(order)
    keep = []

    def dev(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        keep.append(t)
        return t.data_ptr()

    def out(nbytes):
        t = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device="cuda")
        keep.append(t)
        return t.data_ptr()

    cin, cout = (nv.DfdColumn * len(cols))(), (nv.DfdColumn * len(cols))()
    for i, c in enumerate(cols):
        valid = None
        if c["validity"] is not None:
            valid = np.unpackbits(c["validity"], bitorder="little")[:n].astype(bool)[order]
        if c["kind"] == nv.COL_FIXED:
            cin[i] = nv.DfdColumn(c["kind"], c["width"], dev(c["values"][order]), None, dev(bits(valid)) if valid is not None else None, 0, 0)
            cout[i] = nv.DfdColumn(c["kind"], c["width"], out(n * c["width"]), None, out((n + 31) // 32 * 4) if valid is not None else None, 0, 0)
        else:
            lens = np.diff(c["offsets"])[order]
            starts_b = c["offsets"][:-1][order]
            offs = np.r_[0, np.cumsum(lens)].astype(np.int32)
            data = c["values"][np.repeat(starts_b - offs[:-1], lens) + np.arange(int(offs[-1]))]
            cin[i] = nv.DfdColumn(c["kind"], 0, dev(data), dev(offs), dev(bits(valid)) if valid is not None else None, 0, len(data))
            cout[i] = nv.DfdColumn(c["kind"], 0, out(len(data)), out((n + 1) * 4), out((n + 31) // 32 * 4) if valid is not None else None, 0,
                                   max(len(data), 16))
    d_starts = dev(starts)
    k_arr, o_arr = (C.c_int32 * len(keys))(*keys), (C.c_int32 * len(ops))(*ops)
    host = (C.c_int64 * (N + 1))()
    torch.cuda.synchronize()
    L = nv.lib()

    def call():
        nv.check(L.dfd_partial_reduce_device(ctx.handle, cin, len(cols), n, k_arr, len(keys), o_arr, d_starts, N, cout, host, None))

    for _ in range(warmup):
        call()
    ms = []
    for _ in range(iters):
        ctx.timer_start()
        call()
        ms.append(ctx.timer_stop())
    launches_before = ctx.metrics()["kernel_launches"]
    call()
    launches = ctx.metrics()["kernel_launches"] - launches_before
    ms = np.array(ms)
    ctx.close()
    return {"rows": n, "partitions": N, "groups": int(host[N]), "key_columns": len(keys), "columns": len(cols),
            "kernel_launches_per_call": int(launches), "iters": iters, "warmup": warmup,
            "median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()),
            "p10_ms": float(np.percentile(ms, 10)), "p90_ms": float(np.percentile(ms, 90))}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("workloads", nargs="*", metavar="WORKLOAD", help=f"any of {', '.join(WORKLOADS)} (default: all)")
    ap.add_argument("--iters", type=int, default=200, help="timed calls per workload")
    ap.add_argument("--warmup", type=int, default=20, help="untimed calls before the timed ones")
    args = ap.parse_args()
    bad = [w for w in args.workloads if w not in WORKLOADS]
    if bad:
        ap.error(f"unknown workload(s) {', '.join(bad)}; choose from {', '.join(WORKLOADS)}")
    if args.iters < 1 or args.warmup < 0:
        ap.error("--iters must be >= 1 and --warmup >= 0")
    try:
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device")
        import datafusion_distributed_b200 as dfd

        dfd.WorkerContext(0).close()
    except Exception as e:  # noqa: BLE001
        print(f"bench_reduce.py: needs a GPU ({e}); nothing measured", file=sys.stderr)
        return 2
    name, power = gpu_info()
    for w in args.workloads or WORKLOADS:
        r = run(w, args.iters, args.warmup)
        r.update({"workload": w, "gpu": name, "power_limit": power})
        if w == "q1":
            r["median_us"] = r["median_ms"] * 1000.0
        print(json.dumps(r), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
