"""GPU parity tests of the device-side PartialReduce (dfd_partial_reduce_device) against a CPU group-by of the same
partitioned rows.  Integer aggregates (SUM / COUNT / MIN / MAX over i64, SUM over 128-bit decimals) are bit-exact; the
float sum is atomics-ordered, so it is compared with the exact sum of its group within the recursive-summation bound
(k-1) * 2^-53 * sum|x| (tests/test_reduce_exact_gpu.py::assert_float_sum_within_bound)."""
import uuid

import numpy as np
import pandas as pd
import pyarrow as pa
import pytest

import datafusion_distributed_b200 as dfd
from datafusion_distributed_b200 import _native as nv
from oracle import oracle as orc
from tests.test_reduce_exact_gpu import assert_float_sum_within_bound
from tests.util import expected_partitions

pytestmark = pytest.mark.gpu


def make_partial_agg_table(n, n_groups, seed):
    """The output of a Partial aggregate: (g1: Int64, g2: Int32) group keys + states sum_i64, count, min_i64, max_i64, sum_f64,
    sum_dec (Decimal128 as two int64 limbs)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    g1 = rng.integers(0, n_groups, n, dtype=np.int64) * 1_000_003
    g2 = (g1 % 7).astype(np.int32)
    s = rng.integers(-(1 << 40), 1 << 40, n, dtype=np.int64)
    cnt = rng.integers(1, 100, n, dtype=np.int64)
    mn = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)
    mx = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)
    f = rng.standard_normal(n)
    dec = np.zeros((n, 2), dtype=np.int64)
    dec[:, 0] = rng.integers(-(1 << 62), 1 << 62, n, dtype=np.int64)  # low limb with the top bit set half of the time -> carries
    dec[:, 1] = rng.integers(-5, 5, n, dtype=np.int64)
    return g1, g2, s, cnt, mn, mx, f, dec


OPS = [-1, -1, nv.AGG_SUM_I64, nv.AGG_SUM_I64, nv.AGG_MIN_I64, nv.AGG_MAX_I64, nv.AGG_SUM_F64, nv.AGG_SUM_I128]


def dec_to_int(limbs):
    return [(int(hi) << 64) + (int(lo) & ((1 << 64) - 1)) for lo, hi in limbs]


def oracle_groups(cols, rows):
    """CPU PartialReduce of the given rows: {(g1, g2): (sum, count, min, max, float inputs, decsum)}."""
    g1, g2, s, cnt, mn, mx, f, dec = [c[rows] for c in cols]
    df = pd.DataFrame({"g1": g1, "g2": g2, "s": s, "cnt": cnt, "mn": mn, "mx": mx, "f": f})
    df["dec"] = [d - (1 << 128) if d >= (1 << 127) else d for d in [x % (1 << 128) for x in dec_to_int(dec)]]
    out = {}
    for (a, b), grp in df.groupby(["g1", "g2"], sort=False):
        dsum = sum(grp["dec"]) % (1 << 128)
        out[(int(a), int(b))] = (int(np.sum(grp["s"].to_numpy(), dtype=np.int64)), int(grp["cnt"].sum()), int(grp["mn"].min()), int(grp["mx"].max()),
                                 grp["f"].tolist(), dsum)
    return out


def upload(ctx, cols):
    import torch

    keep, dcols = [], []
    for c in cols:
        if c.shape[0] == 0:  # (a zero-element torch tensor has no storage: give the descriptor a real address)
            c = np.zeros((1,) + c.shape[1:], dtype=c.dtype)
        t = torch.from_numpy(np.ascontiguousarray(c)).cuda()
        keep.append(t)
        if c.ndim == 2:
            dcols.append(dfd.DeviceColumn(nv.COL_FIXED, 16, t.data_ptr(), length=c.shape[0], keep=t))
        else:
            dcols.append(dfd.DeviceColumn.from_torch(t))
    torch.cuda.synchronize()
    return dcols, keep


def download(ctx, col, rows, dtype, width_elems=1):
    out = np.empty(rows * width_elems, dtype=dtype)
    if rows:
        nv.check(nv.lib().dfd_memcpy_d2h(ctx.handle, out.ctypes.data, col.values, out.nbytes))
    return out.reshape(rows, width_elems) if width_elems > 1 else out


def check_reduced(ctx, outs, out_starts, cols, dest, N, segs=None):
    dts = [np.int64, np.int32, np.int64, np.int64, np.int64, np.int64, np.float64, np.int64]
    total = int(out_starts[-1])
    host = [download(ctx, outs[i], total, dts[i], 2 if i == 7 else 1) for i in range(8)]
    for p in range(N):
        want = oracle_groups(cols, np.nonzero(dest == p)[0])
        a, b = int(out_starts[p]), int(out_starts[p + 1])
        assert b - a == len(want), (p, b - a, len(want))
        seen = set()
        for r in range(a, b):
            k = (int(host[0][r]), int(host[1][r]))
            assert k in want and k not in seen, (p, k)
            seen.add(k)
            w = want[k]
            assert (int(host[2][r]), int(host[3][r]), int(host[4][r]), int(host[5][r])) == w[:4], (p, k)
            assert_float_sum_within_bound(host[6][r], w[4], (p, k))
            assert ((int(host[7][r][1]) << 64) + (int(host[7][r][0]) & ((1 << 64) - 1))) % (1 << 128) == w[5], (p, k)


@pytest.mark.parametrize("n,n_groups,N", [(0, 1, 4), (1, 1, 1), (5_000, 17, 8), (200_003, 5_000, 12), (300_000, 250_000, 48)])
def test_partial_reduce_matches_cpu_group_by(ctx, n, n_groups, N):
    cols = make_partial_agg_table(n, n_groups, 11)
    dcols, _keep = upload(ctx, cols)
    part = dfd.HashPartitioner(ctx, dfd.Partitioning.Hash([0, 1], N))
    pouts, starts = part.partition(dcols, n)
    red = dfd.PartialReduceExec(ctx, [0, 1], OPS)
    outs, out_starts = red.reduce(pouts, n, part.part_starts_device_ptr(), N)
    dest = orc.partition_ids([cols[0], cols[1]], n, N) if n else np.zeros(0, dtype=np.uint32)
    check_reduced(ctx, outs, out_starts, cols, dest, N)
    assert out_starts[-1] <= n


def test_partial_reduce_then_prepartitioned_shuffle(ctx):
    """Partial output -> repartition -> PartialReduce -> exchange, all on the device (world = 1): partition q's single
    segment holds exactly the reduced groups of destination q."""
    n, N = 120_000, 6
    cols = make_partial_agg_table(n, 3_000, 5)
    dcols, _keep = upload(ctx, cols)
    part = dfd.HashPartitioner(ctx, dfd.Partitioning.Hash([0, 1], N))
    pouts, _ = part.partition(dcols, n)
    outs, out_starts = dfd.PartialReduceExec(ctx, [0, 1], OPS).reduce(pouts, n, part.part_starts_device_ptr(), N)
    ex = dfd.ShuffleExchange(ctx, 0, 1, None)
    ex.setup_window(16 << 20)
    node = dfd.NetworkShuffleExec.try_new(dfd.Partitioning.Hash([0, 1], N), uuid.uuid4(), 1, 1, 1)
    wcols, ss, sc = node.shuffle_partitioned(ex, outs, out_starts)
    assert np.array_equal(sc[:, 0], np.diff(out_starts))
    dest = orc.partition_ids([cols[0], cols[1]], n, N)
    for q in (0, N - 1):
        want = oracle_groups(cols, np.nonzero(dest == q)[0])
        a, cnt = int(ss[q, 0]), int(sc[q, 0])
        g1 = dfd.NetworkShuffleExec.segment_to_arrow(ctx, dfd.DeviceColumn(nv.COL_FIXED, 8, wcols[0].values, arrow_type=pa.int64()), a, cnt).to_numpy()
        sm = dfd.NetworkShuffleExec.segment_to_arrow(ctx, dfd.DeviceColumn(nv.COL_FIXED, 8, wcols[2].values, arrow_type=pa.int64()), a, cnt).to_numpy()
        g2 = dfd.NetworkShuffleExec.segment_to_arrow(ctx, dfd.DeviceColumn(nv.COL_FIXED, 4, wcols[1].values, arrow_type=pa.int32()), a, cnt).to_numpy()
        assert len(g1) == len(want)
        for i in range(len(g1)):
            assert want[(int(g1[i]), int(g2[i]))][0] == int(sm[i])
    ex.close()


def test_partial_reduce_argument_errors(ctx):
    cols = make_partial_agg_table(100, 5, 1)
    dcols, _keep = upload(ctx, cols)
    part = dfd.HashPartitioner(ctx, dfd.Partitioning.Hash([0], 4))
    pouts, _ = part.partition(dcols, 100)
    with pytest.raises(dfd.DfdError):  # a key column that carries an aggregate
        dfd.PartialReduceExec(ctx, [0, 1], [nv.AGG_SUM_I64] + OPS[1:]).reduce(pouts, 100, part.part_starts_device_ptr(), 4)
    with pytest.raises(dfd.DfdError):  # SUM_I128 on an 8-byte column
        dfd.PartialReduceExec(ctx, [0, 1], OPS[:2] + [nv.AGG_SUM_I128] + OPS[3:]).reduce(pouts, 100, part.part_starts_device_ptr(), 4)
