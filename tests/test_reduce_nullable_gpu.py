"""Exact checks of the device-side PartialReduce (dfd_partial_reduce_device) with nullable group keys and states, Utf8 /
LargeUtf8 / Binary group keys and Boolean group keys, against a plain reference of the same operation.

The reference is a Python group-by that extends the one of tests/test_reduce_exact_gpu.py (whose folds it reuses):
  - a key value is its bytes (fixed-width), its bytes (strings), a bool (Boolean) or None (NULL); a group is (input
    partition, tuple of key values), so NULL is a group value, equal to NULL only, and the null pattern of several keys is
    part of the key;
  - a state folds only its non-null inputs (integer ops exactly, float MIN / MAX by totalOrder, float SUM within the
    recursive-summation bound) and is None when every input of its group is null.
The device must write zero bytes under a null key (length 0 for a string, bit 0 for a Boolean) and 0 under a null state.
Tests without a GPU check the reference itself, including against pyarrow's group_by."""
import ctypes as C
import uuid

import numpy as np
import pyarrow as pa
import pytest

import datafusion_distributed_b200 as dfd
from datafusion_distributed_b200 import _native as nv
from tests.test_reduce_exact_gpu import (ALL_OPS, INT64_MAX, INT64_MIN, M64, MAX_F64, MAX_I64, MIN_F64, MIN_I64, SUM_F64, SUM_I64,
                                         SUM_I128, _bits_to_float, _fold, _inputs, _outputs, _special_bits,
                                         assert_float_sum_within_bound, by_destination, state_column)

ERR_INVALID_ARGUMENT, ERR_UNSUPPORTED, ERR_CAPACITY = 1, 6, 7
STRING_KINDS = {"utf8": nv.COL_UTF8, "large_utf8": nv.COL_LARGE_UTF8, "binary": nv.COL_BINARY}


# ------------------------------------------------------------------------------------------------ reference ----

class Col:
    """One column as the reference sees it.  kind: "fixed" (data: (n,) or (n, 2) array), "bool" (data: bool array) or a
    string kind (data: list of bytes); valid: bool array or None (no validity bitmap).  Under a null the data holds
    whatever the test put there."""

    def __init__(self, kind, data, valid=None):
        self.kind, self.data, self.valid = kind, data, None if valid is None else np.asarray(valid, dtype=bool)

    def __len__(self):
        return len(self.data)

    def take(self, order):
        d = [self.data[i] for i in order] if isinstance(self.data, list) else self.data[order]
        return Col(self.kind, d, None if self.valid is None else self.valid[order])

    def is_valid(self, r):
        return self.valid is None or bool(self.valid[r])

    def key_value(self, r):
        if not self.is_valid(r):
            return None
        if self.kind == "fixed":
            return np.ascontiguousarray(self.data[r:r + 1]).tobytes()
        if self.kind == "bool":
            return bool(self.data[r])
        return bytes(self.data[r])


def nullable_reference(cols, key_idx, ops, part_starts):
    """{(input partition, key tuple): [folded state or None (null) per column; None for keys]}."""
    n, N = len(cols[0]), len(part_starts) - 1
    part = np.repeat(np.arange(N), np.diff(np.asarray(part_starts))).tolist()
    assert len(part) == n
    rows = {}
    for r in range(n):
        rows.setdefault((part[r], tuple(cols[k].key_value(r) for k in key_idx)), []).append(r)
    vals = [None if op < 0 else _inputs(op, cols[c].data) for c, op in enumerate(ops)]
    out = {}
    for g, idx in rows.items():
        states = []
        for c, op in enumerate(ops):
            if op < 0:
                states.append(None)
                continue
            live = [vals[c][i] for i in idx if cols[c].is_valid(i)]
            states.append(_fold(op, live) if live else None)
        out[g] = states
    return out


# -------------------------------------------------------------------------------------------- device staging ----

def _pack_bits(bits):
    b = np.packbits(np.asarray(bits, dtype=np.uint8), bitorder="little")
    return np.concatenate([b, np.zeros((-len(b)) % 8 + 8, np.uint8)])  # whole words and some slack


def _unpack_bits(raw, n):
    return np.unpackbits(np.asarray(raw, dtype=np.uint8), bitorder="little")[:n].astype(bool)


class Staged:
    """Device copies of Col inputs at an Arrow `offset` (leading rows of garbage in every buffer; string offsets that start
    past 0), output buffers pre-filled with 0xAB, part_starts and a device out_part_starts."""

    def __init__(self, ctx, cols, ops, part_starts, offset=0, nullable_out=None, rng=None):
        rng = rng or np.random.Generator(np.random.PCG64(1))
        self.ctx, self.cols, self.ops, self.n, self.N = ctx, cols, ops, len(cols[0]), len(part_starts) - 1
        self.keep, self.cin, self.cout, self.outs = [], [], [], []
        n, off = self.n, offset
        for i, col in enumerate(cols):
            validity = None
            if col.valid is not None:
                validity = self._up(_pack_bits(np.r_[rng.random(off) < 0.5, col.valid]))
            if col.kind == "fixed":
                a = np.ascontiguousarray(col.data)
                w = a.dtype.itemsize * (a.shape[1] if a.ndim == 2 else 1)
                raw = np.concatenate([rng.integers(0, 256, off * w, dtype=np.uint8), a.view(np.uint8).reshape(-1)])
                ic = nv.DfdColumn(nv.COL_FIXED, w, self._up(raw), None, validity, off, 0)
                ob = self._out(max(n * w, 16))
                oc = nv.DfdColumn(nv.COL_FIXED, w, ob, None, None, 0, 0)
            elif col.kind == "bool":
                ic = nv.DfdColumn(nv.COL_BOOL, 0, self._up(_pack_bits(np.r_[rng.random(off) < 0.5, col.data])), None, validity, off, 0)
                oc = nv.DfdColumn(nv.COL_BOOL, 0, self._out((n + 31) // 32 * 4 + 4), None, None, 0, 0)
            else:
                kind = STRING_KINDS[col.kind]
                odt = np.int64 if kind == nv.COL_LARGE_UTF8 else np.int32
                lead = [bytes(rng.integers(0, 256, rng.integers(0, 9), dtype=np.uint8)) for _ in range(off)]
                strs = lead + list(col.data)
                first = 5  # the first offset is not 0
                offs = np.r_[0, np.cumsum([len(s) for s in strs])].astype(odt) + first
                data = np.frombuffer(b"\x11" * first + b"".join(strs), dtype=np.uint8)
                ic = nv.DfdColumn(kind, 0, self._up(data), self._up(offs), validity, off, 0)
                cap = sum(len(s) for s in col.data) + 8
                oc = nv.DfdColumn(kind, 0, self._out(cap), self._out((n + 1) * np.dtype(odt).itemsize), None, 0, cap)
            if col.valid is not None or (nullable_out and nullable_out[i]):
                oc.validity = self._out((n + 31) // 32 * 4 + 4)
            self.cin.append(ic)
            self.cout.append(oc)
        self.part_starts = ctx.upload(np.asarray(part_starts, dtype=np.int64))
        self.dev_starts = ctx.alloc(8 * (self.N + 1))
        self.keep += [self.part_starts, self.dev_starts]

    def _up(self, arr):
        b = self.ctx.upload(np.ascontiguousarray(arr))
        self.keep.append(b)
        return b.ptr

    def _out(self, nbytes):
        b = self.ctx.alloc(nbytes)
        nv.check(nv.lib().dfd_memset_device(self.ctx.handle, b.ptr, 0xAB, nbytes))
        self.keep.append(b)
        self.outs.append(b)
        return b.ptr

    def call(self, key_idx, ops=None, cin=None, cout=None, n_rows=None):
        ops = self.ops if ops is None else ops
        cin, cout = cin or self.cin, cout or self.cout
        host = (C.c_int64 * (self.N + 1))()
        rc = nv.lib().dfd_partial_reduce_device(self.ctx.handle, (nv.DfdColumn * len(cin))(*cin), len(cin), self.n if n_rows is None else n_rows,
                                                (C.c_int32 * len(key_idx))(*key_idx), len(key_idx), (C.c_int32 * len(ops))(*ops),
                                                self.part_starts.ptr, self.N, (nv.DfdColumn * len(cout))(*cout), host, self.dev_starts.ptr)
        self.out_starts = np.frombuffer(host, dtype=np.int64).copy()
        return rc

    def _d2h(self, ptr, nbytes, dtype=np.uint8):
        out = np.empty(max(nbytes, 1), dtype=np.uint8)
        if nbytes:
            nv.check(nv.lib().dfd_memcpy_d2h(self.ctx.handle, out.ctypes.data, ptr, nbytes))
        return out[:nbytes].view(dtype)

    def outputs(self):
        """-> per column (values, valid bool array or None): fixed -> array, bool -> bool array, strings -> list of bytes.
        Checks the device out_part_starts and the string layout (offsets[0] = 0, monotone)."""
        total = int(self.out_starts[-1])
        assert np.array_equal(self._d2h(self.dev_starts.ptr, 8 * (self.N + 1), np.int64), self.out_starts)
        res = []
        for col, oc in zip(self.cols, self.cout):
            valid = _unpack_bits(self._d2h(oc.validity, (total + 7) // 8), total) if oc.validity else None
            if col.kind == "fixed":
                a = np.ascontiguousarray(col.data)
                vals = self._d2h(oc.values, total * oc.width).view(a.dtype).reshape((total,) + a.shape[1:])
            elif col.kind == "bool":
                vals = _unpack_bits(self._d2h(oc.values, (total + 7) // 8), total)
            else:
                odt = np.int64 if oc.kind == nv.COL_LARGE_UTF8 else np.int32
                offs = self._d2h(oc.offsets, (total + 1) * np.dtype(odt).itemsize, odt).astype(np.int64)
                assert offs[0] == 0 and np.all(np.diff(offs) >= 0), "string offsets start at 0 and are monotone"
                raw = self._d2h(oc.values, int(offs[-1])).tobytes()
                vals = [raw[offs[r]:offs[r + 1]] for r in range(total)]
            res.append((vals, valid))
        return res


def check_nullable(st, key_idx):
    """Output partition p holds exactly the groups of input partition p, each once, with exact states; zero bytes under
    null keys and null states.  Returns {(p, key tuple): [states]}."""
    cols, ops = st.cols, st.ops
    part_starts = np.r_[0, np.cumsum(np.diff(st.part_starts.download(np.int64, st.N + 1)))]
    want = nullable_reference(cols, key_idx, ops, part_starts)
    counts = np.zeros(st.N, dtype=np.int64)
    for p, _ in want:
        counts[p] += 1
    assert st.out_starts.tolist() == [0] + np.cumsum(counts).tolist(), "output partition boundaries"
    outs = st.outputs()
    states_out = [None if op < 0 else _outputs(op, outs[c][0]) for c, op in enumerate(ops)]
    got = {}
    for p in range(st.N):
        for r in range(int(st.out_starts[p]), int(st.out_starts[p + 1])):
            key = []
            for k in key_idx:
                vals, valid = outs[k]
                if valid is not None and not valid[r]:
                    zero = {"fixed": lambda: not np.ascontiguousarray(vals[r:r + 1]).view(np.uint8).any(),
                            "bool": lambda: not vals[r]}.get(cols[k].kind, lambda: vals[r] == b"")()
                    assert zero, f"row {r}: bytes under a null key are not zero"
                    key.append(None)
                else:
                    key.append(Col(cols[k].kind, vals).key_value(r))
            g = (p, tuple(key))
            assert g in want, f"output row {r} of partition {p}: key {g[1]} is not a group of input partition {p}"
            assert g not in got, f"output partition {p} holds key {g[1]} twice"
            states = []
            for c, op in enumerate(ops):
                if op < 0:
                    states.append(None)
                    continue
                valid = outs[c][1]
                if valid is not None and not valid[r]:
                    assert want[g][c] is None, (f"partition {p} key {g[1]} column {c}: null, want {want[g][c]}")
                    assert states_out[c][r] == 0, f"partition {p} key {g[1]} column {c}: null state not written as 0"
                    states.append(None)
                    continue
                assert want[g][c] is not None, f"partition {p} key {g[1]} column {c}: want null"
                if op == SUM_F64:
                    assert_float_sum_within_bound(_bits_to_float(states_out[c][r]), want[g][c], (p, g[1], c))
                else:
                    assert states_out[c][r] == want[g][c], (f"partition {p} key {g[1]} column {c} op {op}", states_out[c][r], want[g][c])
                states.append(states_out[c][r])
            got[g] = states
    assert len(got) == len(want)
    return got


def run_check(ctx, cols, key_idx, ops, part_starts, offset=0, nullable_out=None):
    st = Staged(ctx, cols, ops, part_starts, offset, nullable_out)
    nv.check(st.call(key_idx))
    return check_nullable(st, key_idx)


def permuted(cols, order):
    return [c.take(order) for c in cols]


def poisoned_states(op, n, valid, rng):
    """Random state inputs with the values that break a reduce if they leak put under the nulls: NaN and -NaN for floats,
    INT64_MIN / INT64_MAX for integers, all-ones low limbs (a carry) and high limbs for SUM_I128."""
    a = state_column(op, n, rng)
    bad = ~valid
    if op in (SUM_F64, MIN_F64, MAX_F64):
        a.view(np.uint64)[bad] = rng.choice(np.array([0x7FF8_0000_0000_0000, 0xFFF8_0000_0000_0001, 0x7FF0_0000_0000_0000,
                                                      0xFFF0_0000_0000_0000], np.uint64), int(bad.sum()))
    elif op == SUM_I128:
        a[bad] = np.array([M64, M64 >> 1], np.uint64)
    else:
        a[bad] = rng.choice(np.array([INT64_MIN, INT64_MAX], np.int64), int(bad.sum()))
    return a


def random_strings(rng, n, vocab):
    return [vocab[i] for i in rng.integers(0, len(vocab), n)]


# ---------------------------------------------------------------------------------------- reference checks ----

def test_reference_against_pyarrow_group_by():
    """Integer SUM / MIN / MAX with null keys (Utf8, Int32, Boolean) and null states, one partition, against
    pyarrow.Table.group_by(...).aggregate(...): null keys form groups, an all-null group's state is null."""
    rng = np.random.Generator(np.random.PCG64(3))
    n = 3000
    s = random_strings(rng, n, [b"", b"a", b"ab", b"Yes", b"No"])
    sv = rng.random(n) < 0.8
    i32 = rng.integers(-3, 3, n).astype(np.int32)
    iv = rng.random(n) < 0.7
    bl = rng.random(n) < 0.5
    bv = rng.random(n) < 0.9
    ids = rng.integers(0, 40, n)
    vals = [rng.integers(-1000, 1000, n, dtype=np.int64) for _ in range(3)]
    vv = [(rng.random(n) < 0.6) & (ids % 7 != 0) for _ in range(3)]  # ids divisible by 7: every state null
    cols = [Col("utf8", s, sv), Col("fixed", i32, iv), Col("bool", bl, bv)] + [Col("fixed", v, m) for v, m in zip(vals, vv)]
    ops = [-1, -1, -1, SUM_I64, MIN_I64, MAX_I64]
    # the state nulls depend on ids: make ids a key too, through the Int32 column
    cols[1] = Col("fixed", (i32 * 100 + ids).astype(np.int32), iv)
    want = nullable_reference(cols, [0, 1, 2], ops, [0, n])
    t = pa.table({"s": pa.array([x.decode() for x in s], mask=~sv), "i": pa.array(cols[1].data, mask=~iv), "b": pa.array(bl, mask=~bv),
                  "x": pa.array(vals[0], mask=~vv[0]), "y": pa.array(vals[1], mask=~vv[1]), "z": pa.array(vals[2], mask=~vv[2])})
    agg = t.group_by(["s", "i", "b"]).aggregate([("x", "sum"), ("y", "min"), ("z", "max")]).to_pylist()
    assert len(agg) == len(want)
    n_null_groups = 0
    for row in agg:
        k = (0, (None if row["s"] is None else row["s"].encode(),
                 None if row["i"] is None else np.array([row["i"]], np.int32).tobytes(), row["b"]))
        assert want[k][3:] == [row["x_sum"], row["y_min"], row["z_max"]], k
        n_null_groups += None in k[1]
    assert n_null_groups > 10
    assert any(v[3] is None for v in want.values()) and any(v[3] is not None for v in want.values())


def test_reference_null_pattern_and_empty_string_are_distinct_groups():
    cols = [Col("utf8", [b"", b"x", b"", b"zz", b"a"], [False, True, True, False, True]),
            Col("utf8", [b"a", b"a", b"a", b"q", b"a"], [True, True, True, False, True]),
            Col("fixed", np.array([1, 2, 3, 4, 5], np.int64), [True, True, False, False, True])]
    want = nullable_reference(cols, [0, 1], [-1, -1, SUM_I64], [0, 5])
    assert want == {(0, (None, b"a")): [None, None, 1], (0, (b"", b"a")): [None, None, None], (0, (None, None)): [None, None, None],
                    (0, (b"x", b"a")): [None, None, 2], (0, (b"a", b"a")): [None, None, 5]}


def test_reference_skips_poisoned_null_states():
    rng = np.random.Generator(np.random.PCG64(5))
    n = 200
    valid = rng.random(n) < 0.5
    valid[:2] = True
    for op in ALL_OPS:
        a = poisoned_states(op, n, valid, rng)
        want = nullable_reference([Col("fixed", np.zeros(n, np.int64)), Col("fixed", a, valid)], [0], [-1, op], [0, n])
        k = int(valid.sum())
        clean = nullable_reference([Col("fixed", np.zeros(k, np.int64)), Col("fixed", a[valid])], [0], [-1, op], [0, k])
        assert list(want.values())[0][1] == list(clean.values())[0][1], op


# ---------------------------------------------------------------------------------------------- GPU cases ----

def _nullable_fixed(rng, n, width, p_null, domain):
    """Keys from a small domain (0 included, so a zero value and a null are both common), garbage under the nulls."""
    dt = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}
    if width == 16:
        a = np.stack([rng.integers(0, domain, n, dtype=np.uint64), np.zeros(n, np.uint64)], axis=1)
    else:
        a = rng.integers(0, domain, n).astype(dt[width])
    valid = rng.random(n) >= p_null
    g = rng.integers(0, 256, a.nbytes, dtype=np.uint8).view(a.dtype).reshape(a.shape)
    a[~valid] = g[~valid]
    return Col("fixed", a, valid)


@pytest.mark.gpu
def test_nullable_fixed_keys_at_every_width(ctx):
    rng = np.random.Generator(np.random.PCG64(11))
    n, N = 20_000, 3
    keys = [_nullable_fixed(rng, n, w, 0.3, 5) for w in (1, 2, 4, 8, 16)]
    ones = Col("fixed", np.ones(n, np.int64))
    order, starts = by_destination(rng.integers(0, N, n), N, rng)
    for k in range(5):  # one key at a time: 5 values + NULL per partition
        got = run_check(ctx, permuted([keys[k], ones], order), [0], [-1, SUM_I64], starts)
        assert len(got) == N * 6 and sum(1 for g in got if g[1] == (None,)) == N
    got = run_check(ctx, permuted(keys + [ones], order), list(range(5)), [-1] * 5 + [SUM_I64], starts)
    patterns = {tuple(v is None for v in g[1]) for g in got}
    assert len(patterns) == 32  # every null pattern of 5 keys is its own set of groups


@pytest.mark.gpu
def test_nullable_states_every_op_poison_under_nulls_and_row_orders(ctx):
    """All seven ops with nullable states: NaN / INT64_MIN / INT64_MAX / carrying I128 under the nulls must not leak,
    all-null groups come out null with value 0, and float MIN / MAX are bit-identical across three row orders."""
    rng = np.random.Generator(np.random.PCG64(13))
    n, N, G = 30_000, 4, 900
    gid = rng.integers(0, G, n)
    key = Col("fixed", gid.astype(np.int64))
    cols, ops = [key], [-1]
    for op in ALL_OPS:
        valid = (rng.random(n) < 0.6) & (gid % 9 != 0)  # every 9th group: all null
        a = poisoned_states(op, n, valid, rng)
        if op in (MIN_F64, MAX_F64):
            sb = _special_bits(rng, n)
            a.view(np.uint64)[valid] = sb[valid]
        cols.append(Col("fixed", a, valid))
        ops.append(op)
    runs = []
    for run in range(3):
        order, starts = by_destination(gid % N, N, np.random.Generator(np.random.PCG64(500 + run)))
        got = run_check(ctx, permuted(cols, order), [0], ops, starts)
        runs.append({g: [s for s, op in zip(v, ops) if op in (MIN_F64, MAX_F64)] for g, v in got.items()})
        assert sum(1 for v in got.values() if all(s is None for s in v[1:])) == len({g for g in range(G) if g % 9 == 0})
    assert runs[0] == runs[1] == runs[2]


def _string_vocab(rng):
    base = [b"", b"a", b"\x00", b"\x00\x00", b"a\x00b", b"prefix", b"prefix-", b"prefix-1", b"prefix-2"]
    for L in (7, 8, 9, 15, 16, 17, 31, 32, 33, 255, 256, 257, 300):  # around the 8 / 16 / 256-byte boundaries
        s = bytes(rng.integers(0, 256, L, dtype=np.uint8))
        base += [s, s[:-1] + bytes([s[-1] ^ 1]), b"\x00" * L, (b"shared" * 60)[:L]]
    return list(dict.fromkeys(base))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["utf8", "large_utf8", "binary"])
def test_string_keys(ctx, kind):
    """Lengths 0 to 300 across the 8 / 16 / 256-byte boundaries, unaligned starts, embedded zero bytes, shared prefixes,
    empty string vs NULL, null rows with a non-zero input length, an Arrow offset and a first offset != 0, and equal
    strings in different partitions (different groups)."""
    rng = np.random.Generator(np.random.PCG64(17))
    vocab = _string_vocab(rng)
    if kind != "binary":
        vocab = [v for v in vocab if _is_utf8(v)]
    n, N = 12_000, 5
    s = random_strings(rng, n, vocab)
    valid = rng.random(n) >= 0.15
    for i in np.flatnonzero(~valid)[::2]:
        s[i] = bytes(rng.integers(1, 256, rng.integers(1, 40), dtype=np.uint8))  # garbage of non-zero length under a null
    cols = [Col(kind, s, valid), Col("fixed", rng.integers(-5, 5, n, dtype=np.int64), rng.random(n) < 0.9)]
    order, starts = by_destination(rng.integers(0, N, n), N, rng)
    got = run_check(ctx, permuted(cols, order), [0], [-1, SUM_I64], starts, offset=37)
    assert sum(1 for g in got if g[1] == (None,)) == N and sum(1 for g in got if g[1] == (b"",)) == N


def _is_utf8(b):
    try:
        b.decode("utf-8")
        return True
    except UnicodeDecodeError:
        return False


@pytest.mark.gpu
def test_string_output_layout_slices_per_partition(ctx):
    """Through the Python operator: HashPartitioner -> PartialReduceExec with the default outputs.  The output offsets
    start at 0 and are monotone, and every partition's slice read with DeviceColumn.to_arrow equals the reference."""
    rng = np.random.Generator(np.random.PCG64(19))
    n, N = 50_000, 7
    words = [f"w{i}-" + "x" * int(rng.integers(0, 40)) for i in range(3000)]
    s = pa.array([words[i] for i in rng.zipf(1.3, n) % len(words)], mask=rng.random(n) < 0.05)
    v = pa.array(rng.integers(-100, 100, n), mask=rng.random(n) < 0.3)
    dcols = [dfd.DeviceColumn.from_arrow(ctx, s), dfd.DeviceColumn.from_arrow(ctx, v)]
    part = dfd.HashPartitioner(ctx, dfd.Partitioning.Hash([0], N))
    pouts, starts = part.partition(dcols, n)
    outs, out_starts = dfd.PartialReduceExec(ctx, [0], [-1, SUM_I64]).reduce(pouts, n, part.part_starts_device_ptr(), N)
    offs = outs[0].keep[-2].download(np.int32, int(out_starts[-1]) + 1)
    assert offs[0] == 0 and np.all(np.diff(offs) >= 0)
    host = [pa.concat_arrays([c.to_arrow(ctx, int(starts[p]), int(starts[p + 1])) for p in range(N)]) for c in pouts]
    for p in range(N):
        a, b = int(starts[p]), int(starts[p + 1])
        t = pa.table({"k": host[0][a:b], "v": host[1][a:b]}).group_by(["k"]).aggregate([("v", "sum")])
        want = dict(zip(t.column("k").to_pylist(), t.column("v_sum").to_pylist()))
        k = outs[0].to_arrow(ctx, int(out_starts[p]), int(out_starts[p + 1])).to_pylist()
        sv = outs[1].to_arrow(ctx, int(out_starts[p]), int(out_starts[p + 1])).to_pylist()
        assert len(k) == len(set(k)) == len(want)
        assert dict(zip(k, sv)) == want, p


@pytest.mark.gpu
def test_boolean_keys_with_a_bit_offset(ctx):
    rng = np.random.Generator(np.random.PCG64(23))
    n, N = 5000, 3
    b = rng.random(n) < 0.5
    bv = rng.random(n) < 0.8
    i = rng.integers(0, 3, n).astype(np.int32)
    cols = [Col("bool", b, bv), Col("fixed", i), Col("fixed", rng.integers(0, 9, n, dtype=np.int64), rng.random(n) < 0.5),
            Col("bool", rng.random(n) < 0.5)]
    order, starts = by_destination(rng.integers(0, N, n), N, rng)
    got = run_check(ctx, permuted(cols[:1] + cols[2:3], order), [0], [-1, MAX_I64], starts, offset=13)
    assert sorted({g[1] for g in got}, key=str) == sorted({(True,), (False,), (None,)}, key=str)
    got = run_check(ctx, permuted(cols, order), [0, 1, 3], [-1, -1, MAX_I64, -1], starts, offset=13)
    assert len(got) == N * 3 * 3 * 2


@pytest.mark.gpu
def test_mixed_keys_eight_keys_thirty_two_columns(ctx):
    """Utf8 + Int32 + Boolean + 16-byte keys (and four more), nullable, among 24 nullable state columns of every op; the
    same rows in a second call with non-null inputs but nullable outputs (every output bit set)."""
    rng = np.random.Generator(np.random.PCG64(29))
    n, N = 20_000, 6
    vocab = [b"", b"A", b"N", b"R", b"F", b"O", b"longer string with spaces"]
    key_pos = [0, 4, 9, 13, 18, 22, 27, 31]
    keys = [Col("utf8", random_strings(rng, n, vocab), rng.random(n) >= 0.1), _nullable_fixed(rng, n, 4, 0.1, 3),
            Col("bool", rng.random(n) < 0.5, rng.random(n) >= 0.1), _nullable_fixed(rng, n, 16, 0.1, 2),
            Col("large_utf8", random_strings(rng, n, vocab[:3]), rng.random(n) >= 0.05), _nullable_fixed(rng, n, 1, 0.05, 2),
            Col("binary", random_strings(rng, n, [b"\x00", b"\x00\x00"]), rng.random(n) >= 0.05), _nullable_fixed(rng, n, 8, 0.05, 2)]
    cols, ops = [None] * 32, [-1] * 32
    for j, c in enumerate(key_pos):
        cols[c] = keys[j]
    for i, c in enumerate([c for c in range(32) if c not in key_pos]):
        ops[c] = ALL_OPS[i % 7]
        valid = rng.random(n) < 0.7
        cols[c] = Col("fixed", poisoned_states(ops[c], n, valid, rng), valid)
    order, starts = by_destination(rng.integers(0, N, n), N, rng)
    cols = permuted(cols, order)
    got = run_check(ctx, cols, key_pos, ops, starts, offset=3)
    assert len(got) > 1000
    plain = [Col(c.kind, c.data) for c in cols]
    got2 = run_check(ctx, plain, key_pos, ops, starts, nullable_out=[True] * 32)
    assert all(s is not None for v in got2.values() for s, op in zip(v, ops) if op >= 0)


def q1_table(n_parts, seed):
    """cfg-3's shape: (l_returnflag, l_linestatus) Utf8 groups A/F, N/F, N/O, R/F per input partition, 4 x Decimal128,
    4 x Int64 and 2 x Float64 states, every state nullable."""
    rng = np.random.Generator(np.random.PCG64(seed))
    groups = [("A", "F"), ("N", "F"), ("N", "O"), ("R", "F")] * n_parts
    n = len(groups)
    arrays = [pa.array([g[0] for g in groups]), pa.array([g[1] for g in groups])]
    host = [Col("utf8", [g[0].encode() for g in groups]), Col("utf8", [g[1].encode() for g in groups])]
    ops = [-1, -1]
    for j in range(10):
        valid = rng.random(n) < 0.7
        if j < 4:
            raw = np.zeros((n, 2), dtype=np.uint64)
            raw[:, 0] = rng.integers(0, 1 << 50, n)
            raw[~valid] = np.array([M64, M64 >> 1], np.uint64)
            arrays.append(pa.Array.from_buffers(pa.decimal128(38, 4), n, [pa.py_buffer(np.packbits(valid, bitorder="little").tobytes()),
                                                                           pa.py_buffer(raw.tobytes())], null_count=int((~valid).sum())))
            host.append(Col("fixed", raw, valid))
            ops.append(SUM_I128)
        elif j < 8:
            a = rng.integers(0, 1 << 40, n, dtype=np.int64)
            arrays.append(pa.array(a, mask=~valid))
            host.append(Col("fixed", a, valid))
            ops.append(SUM_I64)
        else:
            a = rng.standard_normal(n)
            arrays.append(pa.array(a, mask=~valid))
            host.append(Col("fixed", a, valid))
            ops.append(MIN_F64 if j == 8 else MAX_F64)
    return arrays, host, ops


@pytest.mark.gpu
def test_q1_shape_end_to_end_through_the_exchange(ctx):
    """24 rows x 2 Utf8 keys x 10 nullable states: HashPartitioner.partition -> PartialReduceExec.reduce ->
    NetworkShuffleExec.shuffle_partitioned at world 1; every segment equals the reference of its partition."""
    arrays, host, ops = q1_table(6, 3)
    n, N = len(arrays[0]), 3
    dcols = [dfd.DeviceColumn.from_arrow(ctx, a) for a in arrays]
    part = dfd.HashPartitioner(ctx, dfd.Partitioning.Hash([0, 1], N))
    pouts, starts = part.partition(dcols, n)
    outs, out_starts = dfd.PartialReduceExec(ctx, [0, 1], ops).reduce(pouts, n, part.part_starts_device_ptr(), N)
    ex = dfd.ShuffleExchange(ctx, 0, 1, None)
    ex.setup_window(16 << 20)
    node = dfd.NetworkShuffleExec.try_new(dfd.Partitioning.Hash([0, 1], N), uuid.uuid4(), 1, 1, 1)
    wcols, ss, sc = node.shuffle_partitioned(ex, outs, out_starts)
    assert np.array_equal(sc[:, 0], np.diff(out_starts))
    # the reference over the partitioned rows as they came out of the partitioner
    prow = [pa.concat_arrays([c.to_arrow(ctx, int(starts[p]), int(starts[p + 1])) for p in range(N)]) for c in pouts]
    pcols = []
    for j, a in enumerate(prow):
        valid = None if a.null_count == 0 else np.asarray(a.is_valid())
        if j < 2:
            pcols.append(Col("utf8", [x.encode() for x in a.to_pylist()]))
        else:
            pcols.append(Col("fixed", _arrow_fixed(a, host[j].data), valid))
    want = nullable_reference(pcols, [0, 1], ops, starts)
    for q in range(N):
        a, cnt = int(ss[q, 0]), int(sc[q, 0])
        seg = [dfd.NetworkShuffleExec.segment_to_arrow(ctx, w, a, cnt) for w in wcols]
        assert cnt == sum(1 for g in want if g[0] == q)
        for r in range(cnt):
            g = (q, (seg[0][r].as_py().encode(), seg[1][r].as_py().encode()))
            for c in range(2, 12):
                v = seg[c][r]
                if want[g][c] is None:
                    assert not v.is_valid, (g, c)
                    continue
                assert v.is_valid, (g, c)
                got = _outputs(ops[c], _arrow_fixed(seg[c].slice(r, 1), host[c].data))[0]
                assert got == want[g][c], (g, c)
    ex.close()


def _arrow_fixed(arr, like):
    """The value buffer of a fixed-width pyarrow array as a numpy array shaped like `like` (nulls keep their bytes)."""
    w = like.dtype.itemsize * (like.shape[1] if like.ndim == 2 else 1)
    buf = np.frombuffer(arr.buffers()[1], dtype=np.uint8)[arr.offset * w:(arr.offset + len(arr)) * w]
    return buf.view(like.dtype).reshape((len(arr),) + like.shape[1:]).copy()


@pytest.mark.gpu
def test_argument_errors_leave_the_context_usable(ctx):
    rng = np.random.Generator(np.random.PCG64(31))
    n = 400
    cols = [Col("utf8", random_strings(rng, n, [b"abc", b"", b"defgh" * 7]), rng.random(n) < 0.8), Col("bool", rng.random(n) < 0.5),
            Col("fixed", rng.integers(0, 5, n, dtype=np.int64), rng.random(n) < 0.5), Col("large_utf8", random_strings(rng, n, [b"x", b"yy"]))]
    ops = [-1, -1, SUM_I64, -1]
    keys = [0, 1, 3]
    st = Staged(ctx, cols, ops, [0, 150, n])

    def cp(src, **kw):
        d = nv.DfdColumn(src.kind, src.width, src.values, src.offsets, src.validity, src.offset, src.values_bytes)
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    cases = {  # name -> (in cols, out cols, ops, status); key columns 0, 1, 3 unless the ops say otherwise
        "capacity": (st.cin, [cp(st.cout[0], values_bytes=3)] + st.cout[1:], ops, ERR_CAPACITY),
        "op on a string": (st.cin, st.cout, [-1, -1, SUM_I64, SUM_I64], ERR_UNSUPPORTED),
        "op on a Boolean": (st.cin, st.cout, [-1, SUM_I64, SUM_I64, -1], ERR_UNSUPPORTED),
        "Utf8 in, Binary out": (st.cin, [cp(st.cout[0], kind=nv.COL_BINARY)] + st.cout[1:], ops, ERR_UNSUPPORTED),
        "LargeUtf8 in, Utf8 out": (st.cin, st.cout[:3] + [cp(st.cout[3], kind=nv.COL_UTF8)], ops, ERR_UNSUPPORTED),
        "Boolean in, fixed out": (st.cin, [st.cout[0], cp(st.cout[1], kind=nv.COL_FIXED, width=1)] + st.cout[2:], ops, ERR_UNSUPPORTED),
        "nullable key, no out validity": (st.cin, [cp(st.cout[0], validity=None)] + st.cout[1:], ops, ERR_UNSUPPORTED),
        "nullable state, no out validity": (st.cin, st.cout[:2] + [cp(st.cout[2], validity=None)] + st.cout[3:], ops, ERR_UNSUPPORTED),
        "unknown kind": ([cp(st.cin[0], kind=9)] + st.cin[1:], [cp(st.cout[0], kind=9)] + st.cout[1:], ops, ERR_UNSUPPORTED),
        "NULL offsets": ([cp(st.cin[0], offsets=None)] + st.cin[1:], st.cout, ops, ERR_INVALID_ARGUMENT),
    }
    for name, (cin, cout, o, status) in cases.items():
        rc = st.call([k for k in keys if o[k] < 0], o, cin, cout)
        assert rc == status, (name, rc, nv.lib().dfd_last_error())
        if name == "capacity":
            msg = nv.lib().dfd_last_error()
            msg = msg.decode() if isinstance(msg, bytes) else msg
            assert "values_bytes 3 <" in msg, msg
            outs = [st._d2h(st.cout[0].offsets, 16), st._d2h(st.cout[0].validity, 16), st._d2h(st.cout[1].values, 16)]
            assert all((b == 0xAB).all() for b in outs), "a refused call wrote an output column"
        assert nv.check(st.call(keys)) is None, name
        check_nullable(st, keys)


@pytest.mark.gpu
def test_launch_counts_follow_the_header_formula(ctx):
    """4 + F + 4 S launches: F = 1 with a float MIN / MAX column or a MIN / MAX column whose input has validity, S = string
    key columns; nothing for 0 rows (which still writes offsets[0] = 0)."""
    rng = np.random.Generator(np.random.PCG64(37))
    n = 2000
    s1 = Col("utf8", random_strings(rng, n, [b"a", b"bb", b""]), rng.random(n) < 0.9)
    s2 = Col("binary", random_strings(rng, n, [b"\x00", b"z"]))
    k = Col("fixed", rng.integers(0, 4, n).astype(np.int32), rng.random(n) < 0.9)
    b = Col("bool", rng.random(n) < 0.5, rng.random(n) < 0.9)
    nn = lambda a: Col("fixed", a)  # noqa: E731
    nl = lambda a: Col("fixed", a, rng.random(n) < 0.5)  # noqa: E731
    i64 = rng.integers(-9, 9, n, dtype=np.int64)
    f64 = rng.standard_normal(n)
    cases = [  # (cols, keys, ops, launches)
        ([k, nn(i64)], [0], [-1, SUM_I64], 4),
        ([k, nl(i64)], [0], [-1, SUM_I64], 4),
        ([b, nn(i64)], [0], [-1, MIN_I64], 4),
        ([k, nl(i64)], [0], [-1, MIN_I64], 5),
        ([k, nl(i64)], [0], [-1, MAX_I64], 5),
        ([k, nn(f64)], [0], [-1, MAX_F64], 5),
        ([s1, nn(i64)], [0], [-1, SUM_I64], 8),
        ([s1, s2, k, nl(f64), nl(i64)], [0, 1, 2], [-1, -1, -1, MIN_F64, MAX_I64], 13),
    ]
    for cols, keys, ops, launches in cases:
        st = Staged(ctx, cols, ops, [0, n // 3, n])
        before = ctx.metrics()["kernel_launches"]
        nv.check(st.call(keys))
        assert ctx.metrics()["kernel_launches"] - before == launches, ops
        check_nullable(st, keys)
    st = Staged(ctx, [s1, s2, nl(i64)], [-1, -1, SUM_I64], [0, n])
    before = ctx.metrics()["kernel_launches"]
    nv.check(st.call([0, 1], n_rows=0))
    assert ctx.metrics()["kernel_launches"] == before and st.out_starts.tolist() == [0, 0]
    assert st._d2h(st.cout[0].offsets, 4, np.int32)[0] == 0 and st._d2h(st.cout[1].offsets, 4, np.int32)[0] == 0


@pytest.mark.gpu
def test_large_zipf_strings_with_nulls(ctx):
    """2^24 rows of zipf-distributed strings (30 % empty, some NULL) over 16 partitions, COUNT and a nullable SUM,
    checked against a vectorised reference."""
    rng = np.random.Generator(np.random.PCG64(41))
    n, N, V = 1 << 24, 16, 1 << 16
    vocab = [b""] + [b"phrase %d " % i + b"q" * (i % 53) for i in range(1, V)]
    lens = np.array([len(v) for v in vocab], np.int64)
    ids = (rng.zipf(1.2, n) - 1) % V
    ids[rng.random(n) < 0.3] = 0  # empty strings
    valid = rng.random(n) >= 0.02
    ids[~valid] = np.where(rng.random(int((~valid).sum())) < 0.5, 0, 7)  # garbage under the nulls, sometimes "" itself
    gid = np.where(valid, ids, -1)
    dest = (gid * 2_654_435_761 + rng.integers(0, 2, n)) % N  # equal keys in up to two partitions
    order, starts = by_destination(dest, N)
    ids, valid, gid = ids[order], valid[order], gid[order]
    x = rng.integers(-1000, 1000, n, dtype=np.int64)
    xv = rng.random(n) < 0.5
    offs = np.r_[0, np.cumsum(lens[ids])].astype(np.int32)
    blob = np.frombuffer(b"".join(vocab), np.uint8)
    vstart = np.r_[0, np.cumsum(lens)[:-1]]
    data = blob[(np.repeat(vstart[ids] - offs[:-1], lens[ids]) + np.arange(int(offs[-1])))]
    import torch  # device buffers without a Python-level copy of every string

    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    keep = [dev(data), dev(offs), dev(_pack_bits(valid)), dev(np.ones(n, np.int64)), dev(x), dev(_pack_bits(xv)), dev(starts)]
    cin = [nv.DfdColumn(nv.COL_UTF8, 0, keep[0].data_ptr(), keep[1].data_ptr(), keep[2].data_ptr(), 0, len(data)),
           nv.DfdColumn(nv.COL_FIXED, 8, keep[3].data_ptr(), None, None, 0, 0),
           nv.DfdColumn(nv.COL_FIXED, 8, keep[4].data_ptr(), None, keep[5].data_ptr(), 0, 0)]
    obuf = [ctx.alloc(len(data) + 16), ctx.alloc((n + 1) * 4), ctx.alloc(n // 8 + 8), ctx.alloc(n * 8), ctx.alloc(n * 8), ctx.alloc(n // 8 + 8)]
    cout = [nv.DfdColumn(nv.COL_UTF8, 0, obuf[0].ptr, obuf[1].ptr, obuf[2].ptr, 0, len(data) + 16),
            nv.DfdColumn(nv.COL_FIXED, 8, obuf[3].ptr, None, None, 0, 0),
            nv.DfdColumn(nv.COL_FIXED, 8, obuf[4].ptr, None, obuf[5].ptr, 0, 0)]
    torch.cuda.synchronize()
    host = (C.c_int64 * (N + 1))()
    nv.check(nv.lib().dfd_partial_reduce_device(ctx.handle, (nv.DfdColumn * 3)(*cin), 3, n, (C.c_int32 * 1)(0), 1, (C.c_int32 * 3)(-1, SUM_I64, SUM_I64),
                                                keep[6].data_ptr(), N, (nv.DfdColumn * 3)(*cout), host, None))
    out_starts = np.frombuffer(host, np.int64).copy()
    # reference: groups (partition, gid) with gid = -1 for NULL
    part = np.repeat(np.arange(N), np.diff(starts))
    o = np.lexsort((gid, part))
    p_s, g_s = part[o], gid[o]
    first = np.flatnonzero(np.r_[True, (p_s[1:] != p_s[:-1]) | (g_s[1:] != g_s[:-1])])
    want_cnt = np.add.reduceat(np.ones(n, np.int64), first)
    want_sum = np.add.reduceat(np.where(xv, x, 0)[o], first)
    want_sv = np.add.reduceat(xv[o].astype(np.int64), first) > 0
    total = int(out_starts[-1])
    assert total == len(first) and np.array_equal(np.diff(out_starts), np.bincount(p_s[first], minlength=N))
    ooffs = obuf[1].download(np.int32, total + 1).astype(np.int64)
    assert ooffs[0] == 0 and np.all(np.diff(ooffs) >= 0)
    obytes = obuf[0].download(np.uint8, int(ooffs[-1])).tobytes()
    ovalid = _unpack_bits(obuf[2].download(np.uint8, (total + 7) // 8), total)
    index = {v: i for i, v in enumerate(vocab)}
    got_g = np.array([index[obytes[ooffs[r]:ooffs[r + 1]]] if ovalid[r] else -1 for r in range(total)], np.int64)
    assert not any(ooffs[r + 1] != ooffs[r] for r in np.flatnonzero(~ovalid)), "a null key has a non-empty output string"
    got_p = np.repeat(np.arange(N), np.diff(out_starts))
    go = np.lexsort((got_g, got_p))
    assert np.array_equal(got_p[go], p_s[first]) and np.array_equal(got_g[go], g_s[first])
    assert np.array_equal(obuf[3].download(np.int64, total)[go], want_cnt)
    sv = _unpack_bits(obuf[5].download(np.uint8, (total + 7) // 8), total)[go]
    assert np.array_equal(sv, want_sv)
    assert np.array_equal(obuf[4].download(np.int64, total)[go], np.where(want_sv, want_sum, 0))
