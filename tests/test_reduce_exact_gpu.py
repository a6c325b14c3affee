"""Exact checks of the device-side PartialReduce (dfd_partial_reduce_device) against a plain reference of the same
operation, at the widths, values and layouts where a hash aggregate goes wrong.

The reference here never uses the kernel's arithmetic or a dataframe library:
  - integer states are Python ints reduced mod 2^64 (SUM_I64) or 2^128 (SUM_I128) to two's complement;
  - float SUM is checked against math.fsum with the recursive-summation bound |gpu - sum| <= (k-1) * 2^-53 * sum|x| for a
    group of k rows (float_sum_error_bound), because the order in which the atomics land is not fixed;
  - float MIN / MAX are a fold under IEEE-754 totalOrder (Rust's f64::total_cmp, the order arrow's float comparisons use):
    -NaN < -inf < ... < -0.0 < +0.0 < ... < +inf < +NaN, taken through the integer map b ^ ((b >> 63) & 0x7fff..ff) on the
    bit pattern b, and must match bit for bit.
Groups are formed per INPUT partition by key bytes: the same key in two partitions is two groups.  Partitions are built
directly here (rows sorted by a destination chosen in the test, part_starts uploaded as is) so that only the reduce is
under test.  Tests without a GPU check the reference itself."""
import ctypes as C
import math

import numpy as np
import pytest

from datafusion_distributed_b200 import _native as nv

M64 = (1 << 64) - 1
SUM_I64, SUM_F64, MIN_I64, MAX_I64 = nv.AGG_SUM_I64, nv.AGG_SUM_F64, nv.AGG_MIN_I64, nv.AGG_MAX_I64
SUM_I128, MIN_F64, MAX_F64 = nv.AGG_SUM_I128, nv.AGG_MIN_F64, nv.AGG_MAX_F64
ALL_OPS = [SUM_I64, SUM_F64, MIN_I64, MAX_I64, SUM_I128, MIN_F64, MAX_F64]
INT64_MIN, INT64_MAX = -(1 << 63), (1 << 63) - 1
ERR_INVALID_ARGUMENT, ERR_UNSUPPORTED = 1, 6


# ------------------------------------------------------------------------------------------------ reference ----

def wrap64(x):
    return ((x + (1 << 63)) & M64) - (1 << 63)


def total_order_key(bits):
    """Bit patterns of doubles (int64 array) -> int64 whose signed order is IEEE-754 totalOrder.  The map is its own inverse."""
    b = np.asarray(bits).view(np.int64)
    return b ^ ((b >> 63) & 0x7FFF_FFFF_FFFF_FFFF)


def _key_to_bits(k):
    """total_order_key of one Python int, back to the unsigned bit pattern."""
    return (k ^ ((k >> 63) & 0x7FFF_FFFF_FFFF_FFFF)) & M64


def float_sum_error_bound(xs):
    """Bound on |recursive sum - exact sum| of the finite values xs in any order: (k-1) * 2^-53 * sum|x|."""
    return (len(xs) - 1) * 2.0 ** -53 * math.fsum(abs(x) for x in xs)


def assert_float_sum_within_bound(got, xs, what=""):
    """A SUM_F64 result against the exact sum of its group's inputs.  NaN in, or +inf together with -inf, gives NaN;
    otherwise one infinity gives that infinity, and a finite sum is within float_sum_error_bound of math.fsum.  The sign
    of a zero sum is not checked: it depends on the order of the additions."""
    got = float(got)
    if any(math.isnan(x) for x in xs) or (math.inf in xs and -math.inf in xs):
        assert math.isnan(got), (what, got)
    elif math.inf in xs or -math.inf in xs:
        assert got == (math.inf if math.inf in xs else -math.inf), (what, got)
    else:
        err = abs(math.fsum([got] + [-x for x in xs]))  # (got - exact sum), correctly rounded
        bound = float_sum_error_bound(xs)
        assert err <= bound * (1 + 2.0 ** -40), (what, got, math.fsum(xs), err, bound, len(xs))


def width_of(a):
    return a.dtype.itemsize * (a.shape[1] if a.ndim == 2 else 1)


def key_bytes(cols, key_idx):
    """(n, total key width) uint8: the key columns' bytes side by side."""
    n = len(cols[0])
    return np.concatenate([np.ascontiguousarray(cols[k]).view(np.uint8).reshape(n, width_of(cols[k])) for k in key_idx], axis=1)


def _inputs(op, a):
    """One state column's input values in the domain its fold works in."""
    if op in (MIN_F64, MAX_F64):
        return total_order_key(np.ascontiguousarray(a).view(np.int64)).tolist()
    if op == SUM_F64:
        return np.ascontiguousarray(a).view(np.float64).tolist()
    if op == SUM_I128:
        limbs = np.ascontiguousarray(a).view(np.uint64).reshape(-1, 2).tolist()
        return [lo | (hi << 64) for lo, hi in limbs]
    return np.ascontiguousarray(a).view(np.int64).tolist()


def _fold(op, vals):
    if op == SUM_I64:
        return wrap64(sum(vals))
    if op == MIN_I64:
        return min(vals)
    if op == MAX_I64:
        return max(vals)
    if op == SUM_I128:
        return sum(vals) & ((1 << 128) - 1)
    if op == MIN_F64:
        return _key_to_bits(min(vals))
    if op == MAX_F64:
        return _key_to_bits(max(vals))
    return vals  # SUM_F64: the inputs, for assert_float_sum_within_bound


def exact_reference(cols, key_idx, ops, part_starts):
    """{(input partition, key bytes): [folded state of every column (None for keys)]}."""
    n, N = len(cols[0]), len(part_starts) - 1
    part = np.repeat(np.arange(N), np.diff(np.asarray(part_starts))).tolist()
    assert len(part) == n
    kb = key_bytes(cols, key_idx)
    w, raw = kb.shape[1], kb.tobytes()
    rows = {}
    for r in range(n):
        rows.setdefault((part[r], raw[r * w:(r + 1) * w]), []).append(r)
    vals = [None if op < 0 else _inputs(op, cols[c]) for c, op in enumerate(ops)]
    return {g: [None if op < 0 else _fold(op, [vals[c][i] for i in idx]) for c, op in enumerate(ops)] for g, idx in rows.items()}


def _outputs(op, a):
    """A downloaded state column in the domain of _fold's results (floats as bit patterns)."""
    if op in (MIN_F64, MAX_F64, SUM_F64):
        return np.ascontiguousarray(a).view(np.uint64).tolist()
    if op == SUM_I128:
        return [lo | (hi << 64) for lo, hi in np.ascontiguousarray(a).view(np.uint64).reshape(-1, 2).tolist()]
    return np.ascontiguousarray(a).view(np.int64).tolist()


def _bits_to_float(b):
    return float(np.array([b], dtype=np.uint64).view(np.float64)[0])


def check_exact(cols, key_idx, ops, part_starts, outs, out_starts):
    """Output partition p holds exactly the groups of input partition p, each once, with exact states.  Returns
    {(p, key bytes): [state bit patterns]} so that runs can be compared with each other."""
    want = exact_reference(cols, key_idx, ops, part_starts)
    N = len(part_starts) - 1
    counts = np.zeros(N, dtype=np.int64)
    for p, _ in want:
        counts[p] += 1
    assert list(out_starts) == [0] + np.cumsum(counts).tolist(), "output partition boundaries"
    total = int(out_starts[-1])
    kb = key_bytes(outs, key_idx)
    w, raw = kb.shape[1], kb.tobytes()
    got_cols = [None if op < 0 else _outputs(op, outs[c]) for c, op in enumerate(ops)]
    got = {}
    for p in range(N):
        for r in range(int(out_starts[p]), int(out_starts[p + 1])):
            g = (p, raw[r * w:(r + 1) * w])
            assert g in want, f"output row {r} of partition {p}: key {g[1].hex()} is not a group of input partition {p}"
            assert g not in got, f"output partition {p} holds key {g[1].hex()} twice"
            states = [None if op < 0 else got_cols[c][r] for c, op in enumerate(ops)]
            for c, op in enumerate(ops):
                if op == SUM_F64:
                    assert_float_sum_within_bound(_bits_to_float(states[c]), want[g][c], (p, g[1].hex(), c))
                elif op >= 0:
                    assert states[c] == want[g][c], (f"partition {p} key {g[1].hex()} column {c} op {op}", states[c], want[g][c])
            got[g] = states
    assert len(got) == total == len(want)
    return got


def reduce_reference_np(key, part, cols, ops):
    """Vectorised reference for one int64 key column (the large case): rows grouped by (partition, key), groups sorted by
    (partition, key).  Returns (part, key, [state column per op]); SUM_I128 as (n, 2) uint64 limbs, floats as bit patterns."""
    order = np.lexsort((key, part))
    k, p = key[order], part[order]
    first = np.flatnonzero(np.r_[True, (k[1:] != k[:-1]) | (p[1:] != p[:-1])]) if len(k) else np.zeros(0, np.int64)
    states = []
    for a, op in zip(cols, ops):
        a = a[order]
        if op == SUM_I64:
            states.append(np.add.reduceat(a.view(np.uint64), first).view(np.int64))
        elif op in (MIN_I64, MAX_I64):
            states.append((np.minimum if op == MIN_I64 else np.maximum).reduceat(a.view(np.int64), first))
        elif op in (MIN_F64, MAX_F64):
            t = (np.minimum if op == MIN_F64 else np.maximum).reduceat(total_order_key(a.view(np.int64)), first)
            states.append(total_order_key(t).view(np.uint64))
        elif op == SUM_I128:
            limbs = a.view(np.uint64).reshape(-1, 2)
            lo_lo = np.add.reduceat(limbs[:, 0] & np.uint64(0xFFFF_FFFF), first)  # < 2^32 * rows: no wrap
            lo_hi = np.add.reduceat(limbs[:, 0] >> np.uint64(32), first)
            mid = lo_hi + (lo_lo >> np.uint64(32))                                 # the low limb's sum = mid * 2^32 + low 32 bits
            low = (mid << np.uint64(32)) | (lo_lo & np.uint64(0xFFFF_FFFF))
            high = np.add.reduceat(limbs[:, 1], first) + (mid >> np.uint64(32))    # carries out of the low limb
            states.append(np.stack([low, high], axis=1))
        else:
            raise ValueError(f"op {op} has no vectorised reference")
    return p[first], k[first], states


# ---------------------------------------------------------------------------------------- white-box hash copy ----
# Mirrors key_hash in datafusion_distributed_b200/csrc/dfd_reduce.cu for ONE 8-byte key: mix64(0x9e3779b97f4a7c15 ^ key).
# A row of input partition p starts probing at (key_hash + p * 0x9e3779b97f4a7c15) & table_mask, i.e. at key_hash for
# partition 0; the table has the smallest power of two >= max(64, 2 n) slots.

HASH_SEED = 0x9E3779B97F4A7C15
_C1, _C2 = 0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53


def mix64(x):
    x ^= x >> 33
    x = (x * _C1) & M64
    x ^= x >> 33
    x = (x * _C2) & M64
    return x ^ (x >> 33)


def unmix64(x):
    x ^= x >> 33  # (a shift by 33 of 64 bits undoes itself)
    x = (x * pow(_C2, -1, 1 << 64)) & M64
    x ^= x >> 33
    x = (x * pow(_C1, -1, 1 << 64)) & M64
    return x ^ (x >> 33)


def table_slots(n_rows):
    return max(64, 1 << (2 * n_rows - 1).bit_length())


def key_for_slot(slot, slots, r):
    """An int64 key whose key_hash lands on `slot` of a `slots`-slot table (r picks one of the many)."""
    h = ((r << (slots.bit_length() - 1)) | slot) & M64
    return wrap64(unmix64(h) ^ HASH_SEED)


# -------------------------------------------------------------------------------------------- device calls ----

def by_destination(dest, N, rng=None):
    """Row order that sorts rows by destination (shuffled inside each partition with rng) and part_starts[N+1]."""
    dest = np.asarray(dest)
    order = np.lexsort((rng.random(len(dest)), dest)) if rng is not None else np.argsort(dest, kind="stable")
    starts = np.zeros(N + 1, dtype=np.int64)
    starts[1:] = np.cumsum(np.bincount(dest, minlength=N))
    return order, starts


def _call(ctx, cin, n_rows, key_idx, ops, part_starts_ptr, N, cout, host_starts, dev_starts_ptr):
    n_cols = len(cin)
    return nv.lib().dfd_partial_reduce_device(ctx.handle, (nv.DfdColumn * n_cols)(*cin), n_cols, n_rows,
                                              (C.c_int32 * len(key_idx))(*key_idx), len(key_idx), (C.c_int32 * len(ops))(*ops),
                                              part_starts_ptr, N, (nv.DfdColumn * len(cout))(*cout), host_starts, dev_starts_ptr)


class Staged:
    """Input columns (optionally a slice at Arrow `offset` of a longer device column whose leading rows would change the
    result if read), output columns, part_starts and a device out_part_starts, all on the device."""

    def __init__(self, ctx, cols, ops, part_starts, offsets=None):
        self.ctx, self.cols, self.n, self.N = ctx, cols, len(cols[0]), len(part_starts) - 1
        self.keep, self.out_bufs, self.cin, self.cout = [], [], [], []
        for i, a in enumerate(cols):
            a = np.ascontiguousarray(a)
            off = offsets[i] if offsets else 0
            if off:
                if ops[i] < 0:
                    lead = a[np.arange(off) % max(self.n, 1)]  # real keys: read by mistake they would join real groups
                else:
                    lead = np.full(off * width_of(a), 0xFF, dtype=np.uint8).view(a.dtype).reshape((off,) + a.shape[1:])
                a = np.concatenate([lead, a])
            w = width_of(a)
            b = ctx.upload(a)
            o = ctx.alloc(max(self.n * w, 16))
            nv.check(nv.lib().dfd_memset_device(ctx.handle, o.ptr, 0xAB, o.nbytes))
            self.keep.append(b)
            self.out_bufs.append(o)
            self.cin.append(nv.DfdColumn(nv.COL_FIXED, w, b.ptr, None, None, off, 0))
            self.cout.append(nv.DfdColumn(nv.COL_FIXED, w, o.ptr, None, None, 0, 0))
        self.part_starts = ctx.upload(np.asarray(part_starts, dtype=np.int64))
        self.dev_starts = ctx.alloc(8 * (self.N + 1))
        self.keep += [self.part_starts, self.dev_starts]

    def call(self, key_idx, ops):
        """-> status of dfd_partial_reduce_device; on success self.out_starts holds the host out_part_starts."""
        nv.check(nv.lib().dfd_memset_device(self.ctx.handle, self.dev_starts.ptr, 0xAB, self.dev_starts.nbytes))
        host = (C.c_int64 * (self.N + 1))()
        rc = _call(self.ctx, self.cin, self.n, key_idx, ops, self.part_starts.ptr, self.N, self.cout, host, self.dev_starts.ptr)
        self.out_starts = np.frombuffer(host, dtype=np.int64).copy()
        return rc

    def outputs(self):
        """Downloaded output rows [0, out_starts[N]) of every column; checks the device out_part_starts = the host copy."""
        assert np.array_equal(self.dev_starts.download(np.int64, self.N + 1), self.out_starts), "device out_part_starts != host copy"
        total = int(self.out_starts[-1])
        outs = []
        for a, o in zip(self.cols, self.out_bufs):
            elems = a.shape[1] if a.ndim == 2 else 1
            outs.append(o.download(a.dtype, total * elems).reshape((total,) + a.shape[1:]))
        return outs


def reduce_device(ctx, cols, key_idx, ops, part_starts, offsets=None):
    st = Staged(ctx, cols, ops, part_starts, offsets)
    nv.check(st.call(key_idx, ops))
    return st.outputs(), st.out_starts


def run_and_check(ctx, cols, key_idx, ops, part_starts, offsets=None):
    outs, out_starts = reduce_device(ctx, cols, key_idx, ops, part_starts, offsets)
    return check_exact(cols, key_idx, ops, part_starts, outs, out_starts)


def state_column(op, n, rng):
    """Random inputs of one state column."""
    if op == SUM_I128:
        return rng.integers(0, 1 << 64, (n, 2), dtype=np.uint64)
    if op in (SUM_F64, MIN_F64, MAX_F64):
        return rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4, n)
    return rng.integers(INT64_MIN, INT64_MAX, n, dtype=np.int64, endpoint=True)


def permuted(cols, order):
    return [c[order] for c in cols]


# ---------------------------------------------------------------------------------------- reference checks ----

def test_total_order_key_is_ieee_total_order():
    bits = np.array([0xFFF8_0000_0000_0001, 0xFFF8_0000_0000_0000, 0xFFF0_0000_0000_0001, 0xFFF0_0000_0000_0000,  # -NaNs, -inf
                     0xC000_0000_0000_0000, 0x8000_0000_0000_0001, 0x8000_0000_0000_0000,  # -2.0, -min subnormal, -0.0
                     0x0000_0000_0000_0000, 0x0000_0000_0000_0001, 0x3FF0_0000_0000_0000,  # +0.0, +min subnormal, 1.0
                     0x7FF0_0000_0000_0000, 0x7FF0_0000_0000_0001, 0x7FF8_0000_0000_0000, 0x7FFF_FFFF_FFFF_FFFF], dtype=np.uint64)
    k = total_order_key(bits.view(np.int64))
    assert np.all(np.diff(k) > 0)
    assert np.array_equal(total_order_key(k).view(np.uint64), bits)
    assert [_key_to_bits(int(x)) for x in k] == bits.tolist()


def test_mix64_inverse_and_crafted_slots():
    rng = np.random.Generator(np.random.PCG64(3))
    for x in rng.integers(0, 1 << 64, 1000, dtype=np.uint64).tolist() + [0, 1, M64]:
        assert unmix64(mix64(x)) == x and mix64(unmix64(x)) == x
    slots = table_slots(3000)
    assert slots == 8192 and table_slots(1) == 64 and table_slots(32) == 64 and table_slots(33) == 128
    for r in range(1, 50):
        k = key_for_slot(slots - 1, slots, r)
        assert mix64(HASH_SEED ^ (k & M64)) & (slots - 1) == slots - 1


def test_float_sum_bound_is_tight_enough_to_catch_a_lost_row():
    xs = [1.0] * 1000 + [2.0 ** -20]
    assert_float_sum_within_bound(math.fsum(xs), xs)
    with pytest.raises(AssertionError):
        assert_float_sum_within_bound(1000.0, xs)  # the small row dropped
    assert_float_sum_within_bound(float("nan"), [1.0, math.inf, -math.inf])
    with pytest.raises(AssertionError):
        assert_float_sum_within_bound(0.0, [math.nan, 0.0])


def test_vectorised_reference_matches_the_exact_one():
    rng = np.random.Generator(np.random.PCG64(21))
    n, N = 5000, 7
    ops = [SUM_I64, MIN_I64, MAX_I64, SUM_I128, MIN_F64, MAX_F64]
    key = rng.integers(0, 300, n, dtype=np.int64) << 40
    dest = rng.integers(0, N, n)
    vals = [state_column(op, n, rng) for op in ops]
    vals[3][:, 0] = M64 - rng.integers(0, 3, n, dtype=np.uint64)  # carries on every add
    vals[4][::5] = np.nan
    order, starts = by_destination(dest, N)
    cols = permuted([key] + vals, order)
    want = exact_reference(cols, [0], [-1] + ops, starts)
    part = np.repeat(np.arange(N), np.diff(starts))
    p, k, states = reduce_reference_np(cols[0], part, cols[1:], ops)
    assert len(p) == len(want)
    for i in range(len(p)):
        g = (int(p[i]), int(k[i]).to_bytes(8, "little", signed=True))
        got = [None] + [_outputs(op, s[i:i + 1])[0] for op, s in zip(ops, states)]
        assert got == want[g], g


# ---------------------------------------------------------------------------------------------- GPU cases ----

def _top_byte_flip(a, rows):
    """Flip the most significant byte of rows of one key column (little endian: the last byte of the value)."""
    b = a.view(np.uint8).reshape(len(a), -1)
    b[rows, -1] ^= 0x80


@pytest.mark.gpu
def test_every_op_at_every_key_width_with_max_keys_and_columns(ctx):
    """8 keys of 1, 2, 4, 8 and 16 bytes spread among 24 state columns (32 columns), every op at least three times.
    Sibling groups differ from a base group only in the top byte of one key column, or only in one key column."""
    rng = np.random.Generator(np.random.PCG64(101))
    key_pos = [0, 5, 9, 13, 17, 21, 26, 31]
    widths = [1, 2, 4, 8, 16, 16, 8, 4]
    dt = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}
    n_base = 400
    base = [rng.integers(0, 1 << 64, (n_base, 2), dtype=np.uint64) if w == 16 else rng.integers(0, 1 << (8 * w), n_base, dtype=dt[w])
            for w in widths]
    variants = [[b.copy() for b in base]]
    for j in range(8):  # top byte of key j flipped / key j alone replaced, for a quarter of the base groups each
        pick = rng.choice(n_base, n_base // 4, replace=False)
        v = [b[pick].copy() for b in base]
        _top_byte_flip(v[j], np.arange(len(pick)))
        variants.append(v)
        v = [b[pick].copy() for b in base]
        v[j] = v[j] + (np.array([[1, 0]], dtype=np.uint64) if widths[j] == 16 else dt[widths[j]](1))
        variants.append(v)
    keys = [np.concatenate([v[j] for v in variants]) for j in range(8)]
    n_groups = len(keys[0])
    assert len(np.unique(key_bytes(keys, range(8)).view(np.dtype((np.void, sum(widths)))))) == n_groups
    sizes = rng.integers(1, 12, n_groups)
    gid = np.repeat(np.arange(n_groups), sizes)
    n, N = len(gid), 5
    ops = [-1] * 32
    state_pos = [c for c in range(32) if c not in key_pos]
    for i, c in enumerate(state_pos):
        ops[c] = ALL_OPS[i % 7]
    cols = [None] * 32
    for j, c in enumerate(key_pos):
        cols[c] = keys[j][gid]
    for c in state_pos:
        cols[c] = state_column(ops[c], n, rng)
    order, starts = by_destination((gid * 2_654_435_761) % N, N, rng)  # a group stays in one partition
    cols = permuted(cols, order)
    got = run_and_check(ctx, cols, key_pos, ops, starts)
    assert len(got) == n_groups


@pytest.mark.gpu
def test_integer_edges_wrap_and_extremes(ctx):
    """SUM_I64 over thousands of rows near +-2^62 wraps; MIN / MAX see INT64_MIN / INT64_MAX, including one-row groups
    whose only value is the kernel's initial state; SUM_I128 with low limbs 2^64-1, high limbs -2^63 (= 2^63 mod 2^64),
    sums that wrap mod 2^128 and one group of 10^5 rows whose carries all land on one high word."""
    rng = np.random.Generator(np.random.PCG64(7))
    spec = []  # (rows, sum_i64, min_i64, max_i64, sum_i128 limbs)

    def add(k, s, mn, mx, dec):
        spec.append((k, np.broadcast_to(np.asarray(s, np.int64), (k,)), np.broadcast_to(np.asarray(mn, np.int64), (k,)),
                     np.broadcast_to(np.asarray(mx, np.int64), (k,)), np.broadcast_to(np.asarray(dec, np.uint64), (k, 2))))

    near = lambda k, sign: sign * ((1 << 62) - rng.integers(0, 1 << 20, k, dtype=np.int64))  # noqa: E731
    add(4000, near(4000, 1), near(4000, 1), near(4000, -1), [M64, 1 << 63])
    add(3000, near(3000, -1), near(3000, -1), near(3000, 1), np.stack([rng.integers(0, 1 << 64, 3000, dtype=np.uint64),
                                                                        np.full(3000, 1 << 63, dtype=np.uint64)], axis=1))
    add(1, INT64_MAX, INT64_MAX, INT64_MIN, [M64, M64])          # MIN of INT64_MAX alone, MAX of INT64_MIN alone
    add(1, INT64_MIN, INT64_MIN, INT64_MAX, [0, 1 << 63])
    ext = rng.integers(INT64_MIN, INT64_MAX, 500, dtype=np.int64)
    ext[[3, 200]] = INT64_MIN
    ext[[7, 499]] = INT64_MAX
    add(500, ext, ext, ext, np.stack([np.full(500, M64, np.uint64), np.full(500, M64 >> 1, np.uint64)], axis=1))  # 2^127-1 each
    add(2, [INT64_MAX, 1], [INT64_MAX, INT64_MAX], [INT64_MIN, INT64_MIN], [[M64, M64], [1, 0]])  # -1 + 1 = 0 mod 2^128
    big = 100_000
    add(big, rng.integers(1 << 61, 1 << 62, big, dtype=np.int64), rng.integers(INT64_MIN, INT64_MAX, big, dtype=np.int64),
        rng.integers(INT64_MIN, INT64_MAX, big, dtype=np.int64),
        np.stack([M64 - rng.integers(0, 1 << 20, big, dtype=np.uint64), rng.integers(0, 1 << 64, big, dtype=np.uint64)], axis=1))
    gid = np.concatenate([np.full(s[0], g) for g, s in enumerate(spec)])
    key = (gid.astype(np.int64) - 3) * (1 << 61)  # keys that differ in the top bits only
    cols = [key] + [np.concatenate([s[j] for s in spec]) for j in range(1, 5)]
    ops = [-1, SUM_I64, MIN_I64, MAX_I64, SUM_I128]
    N = 3
    order, starts = by_destination(gid % N, N, rng)
    cols = permuted(cols, order)
    got = run_and_check(ctx, cols, [0], ops, starts)
    assert len(got) == len(spec)


def _float_sum_groups(rng):
    groups = []
    for k in rng.integers(1, 400, 150):
        groups.append(rng.standard_normal(k) * 10.0 ** rng.integers(-8, 9))
    for k in (2, 50, 2000):  # heavy cancellation: +-big pairs around a small remainder
        big = rng.standard_normal(k) * 1e15
        groups.append(np.concatenate([big, -big, rng.standard_normal(7) * 1e-3]))
    groups.append(np.array([1e16, 1.0, -1e16, 1.0, 3e-5]))
    groups.append(rng.standard_normal(5000) * 1e300)  # no overflow: |sum| stays far below 1.8e308
    groups.append(np.array([np.inf, 1.0, -np.inf]))
    groups.append(np.array([np.inf, 2.0, np.inf]))
    groups.append(np.array([-np.inf]))
    groups.append(np.array([1.0, np.nan, 2.0]))
    groups.append(np.array([-0.0, -0.0, 0.0]))       # zero sum: sign left unchecked
    groups.append(np.array([-0.0]))
    groups.append(np.array([5e-324, -5e-324, 5e-324]))
    return groups


@pytest.mark.gpu
def test_float_sum_within_the_recursive_summation_bound(ctx):
    rng = np.random.Generator(np.random.PCG64(17))
    groups = _float_sum_groups(rng)
    gid = np.concatenate([np.full(len(g), i) for i, g in enumerate(groups)])
    vals = np.concatenate(groups)
    N = 3
    order, starts = by_destination(gid % N, N, rng)
    cols = permuted([gid.astype(np.int64), vals, vals.copy()], order)
    got = run_and_check(ctx, cols, [0], [-1, SUM_F64, SUM_F64], starts)
    assert len(got) == len(groups)


def _special_bits(rng, k):
    pool = np.array([0x0000_0000_0000_0000, 0x8000_0000_0000_0000, 0x7FF0_0000_0000_0000, 0xFFF0_0000_0000_0000,  # +-0, +-inf
                     0x0000_0000_0000_0001, 0x8000_0000_0000_0001, 0x000F_FFFF_FFFF_FFFF, 0x800A_BCDE_F012_3456,  # subnormals
                     0x7FF8_0000_0000_0000, 0xFFF8_0000_0000_0000, 0x7FF0_0000_0000_0001, 0xFFF0_0000_DEAD_BEEF,  # NaNs
                     0x7FFF_FFFF_FFFF_FFFF, 0xFFFF_FFFF_FFFF_FFFF, 0x7FF4_0000_0000_1234, 0x3FF0_0000_0000_0000,
                     0xBFF0_0000_0000_0000], dtype=np.uint64)
    bits = np.where(rng.random(k) < 0.5, pool[rng.integers(0, len(pool), k)], rng.standard_normal(k).view(np.uint64))
    return bits


def _minmax_groups(rng):
    nan_pos = np.array([0x7FF8_0000_0000_0000, 0x7FF0_0000_0000_0001, 0x7FFF_FFFF_FFFF_FFFF, 0x7FF4_0000_0000_1234], np.uint64)
    nan_neg = nan_pos | np.uint64(1 << 63)
    groups = [
        ("all +NaN", np.tile(nan_pos, 64)),
        ("all NaN, both signs", np.tile(np.concatenate([nan_pos, nan_neg]), 64)),
        ("all -0.0", np.full(500, 1 << 63, np.uint64)),
        ("mixed zeros", np.tile(np.array([0, 1 << 63], np.uint64), 500)),
        ("one +0.0", np.zeros(1, np.uint64)),
        ("-0.0 after many +0.0", np.r_[np.zeros(999, np.uint64), np.uint64(1 << 63)]),
        ("+-inf", np.tile(np.array([0x7FF0_0000_0000_0000, 0xFFF0_0000_0000_0000], np.uint64), 300)),
        ("subnormals", np.array([1, 2, 0x8000_0000_0000_0001, 0x000F_FFFF_FFFF_FFFF, 0x800F_FFFF_FFFF_FFFF], np.uint64)),
    ]
    for i, k in enumerate(rng.integers(1, 300, 120)):
        groups.append((f"random {i}", _special_bits(rng, k)))
    return groups


@pytest.mark.gpu
def test_float_min_max_total_order_and_bit_identical_across_row_orders(ctx):
    """Results equal the totalOrder fold bit for bit (so an all-NaN group gives a NaN, and a group of +0.0 and -0.0 gives
    -0.0 / +0.0), and three runs with the rows permuted inside each partition agree bit for bit."""
    rng = np.random.Generator(np.random.PCG64(23))
    groups = _minmax_groups(rng)
    gid = np.concatenate([np.full(len(b), i) for i, (_, b) in enumerate(groups)])
    bits = np.concatenate([b for _, b in groups])
    N = 4
    dest = gid % N
    runs = []
    for run in range(3):
        order, starts = by_destination(dest, N, np.random.Generator(np.random.PCG64(1000 + run)))
        cols = permuted([gid.astype(np.int64), bits, bits], order)  # (bit patterns: no NaN passes through a float register)
        got = run_and_check(ctx, cols, [0], [-1, MIN_F64, MAX_F64], starts)
        runs.append(got)
    assert runs[0] == runs[1] == runs[2]
    named = {name: i for i, (name, _) in enumerate(groups)}

    def state(name):
        i = named[name]
        return runs[0][(i % N, int(i).to_bytes(8, "little"))][1:]

    assert state("all -0.0") == [1 << 63, 1 << 63]
    assert state("mixed zeros") == [1 << 63, 0]
    assert state("all +NaN") == [0x7FF0_0000_0000_0001, 0x7FFF_FFFF_FFFF_FFFF]
    assert state("all NaN, both signs") == [0xFFFF_FFFF_FFFF_FFFF, 0x7FFF_FFFF_FFFF_FFFF]


@pytest.mark.gpu
def test_float_min_max_launch_count(ctx):
    """The float MIN / MAX states are finished by one extra pass over the output rows, launched only when such a column
    exists."""
    n = 1000
    key = np.arange(n, dtype=np.int64) % 10
    starts = np.array([0, n], dtype=np.int64)
    for ops, launches in (([-1, SUM_I64], 4), ([-1, MIN_F64], 5), ([-1, MAX_F64, MIN_F64], 5)):
        cols = [key] + [np.linspace(-1, 1, n) if op in (MIN_F64, MAX_F64) else np.ones(n, np.int64) for op in ops[1:]]
        st = Staged(ctx, cols, ops, starts)
        before = ctx.metrics()["kernel_launches"]
        nv.check(st.call([0], ops))
        assert ctx.metrics()["kernel_launches"] - before == launches, ops
        check_exact(cols, [0], ops, starts, st.outputs(), st.out_starts)


@pytest.mark.gpu
def test_float_group_keys_are_compared_by_bits(ctx):
    """+0.0, -0.0 and NaNs with different payloads or signs are different groups (key equality is byte equality, i.e.
    f64::to_bits equality)."""
    distinct = np.array([0, 1 << 63, 0x7FF8_0000_0000_0000, 0xFFF8_0000_0000_0000, 0x7FF8_0000_0000_0001, 0x7FF0_0000_0000_0001,
                         0x3FF0_0000_0000_0000, 0x7FF0_0000_0000_0000], dtype=np.uint64)
    rng = np.random.Generator(np.random.PCG64(5))
    reps = rng.integers(1, 50, len(distinct))
    kbits = np.repeat(distinct, reps)
    f32 = np.repeat(np.array([0, 0x8000_0000, 0x7FC0_0000, 0xFFC0_0000, 0x7FC0_0001, 0x7F80_0001, 0x3F80_0000, 0x7F80_0000],
                             dtype=np.uint32), reps)
    n, N = len(kbits), 2
    order, starts = by_destination(np.zeros(n, np.int64), N, rng)
    for keys in ([kbits], [f32], [kbits, f32]):  # f64 / f32 keys as their bit patterns
        cols = permuted(keys + [np.ones(n, np.int64)], order)
        ops = [-1] * len(keys) + [SUM_I64]
        got = run_and_check(ctx, cols, list(range(len(keys))), ops, starts)
        assert len(got) == len(distinct)
        assert sorted(s[-1] for s in got.values()) == sorted(reps.tolist())


@pytest.mark.gpu
def test_hash_table_probe_chains_wrap_to_slot_zero(ctx):
    """White box: mirrors key_hash in dfd_reduce.cu (see the copy above).  Hundreds of distinct keys all start probing at
    the LAST slot of the table the kernel picks, so their chains wrap to slot 0, where further keys start and collide
    with them; the rest are keys at random slots."""
    rng = np.random.Generator(np.random.PCG64(31))
    n_chain, n_low, n_rand = 600, 150, 1500
    n = 2 * n_chain + 2 * n_low + n_rand
    slots = table_slots(n)
    chain = [key_for_slot(slots - 1, slots, r) for r in rng.integers(1, 1 << 40, n_chain).tolist()]
    low = [key_for_slot(int(s), slots, r) for s, r in zip(rng.integers(0, 200, n_low), rng.integers(1, 1 << 40, n_low).tolist())]
    assert all(mix64(HASH_SEED ^ (k & M64)) & (slots - 1) == slots - 1 for k in chain)
    key = np.array(chain * 2 + low * 2 + rng.integers(INT64_MIN, INT64_MAX, n_rand, dtype=np.int64).tolist(), dtype=np.int64)
    assert len(key) == n and table_slots(len(key)) == slots
    perm = rng.permutation(n)
    ops = [-1, SUM_I64, MIN_F64, SUM_I128]
    cols = [key[perm]] + [state_column(op, n, rng) for op in ops[1:]]
    got = run_and_check(ctx, cols, [0], ops, np.array([0, n], dtype=np.int64))
    assert len(got) == len(np.unique(key))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["one group", "every row its own group"])
def test_hash_table_extreme_cardinalities(ctx, case):
    """All rows in one group (every atomic on one output row), and 2^16 distinct keys in a 2^17-slot table (load factor 0.5)."""
    rng = np.random.Generator(np.random.PCG64(41))
    if case == "one group":
        n = 300_000
        key = np.full(n, 0x0123_4567_89AB_CDEF, dtype=np.int64)
    else:
        n = 1 << 16
        key = rng.permutation(np.arange(n, dtype=np.int64) * 0x1_0000_0001)
        assert table_slots(n) == 2 * n
    ops = [-1] + ALL_OPS
    cols = [key] + [state_column(op, n, rng) for op in ALL_OPS]
    got = run_and_check(ctx, cols, [0], ops, np.array([0, n], dtype=np.int64))
    assert len(got) == (1 if case == "one group" else n)


def _layout(case, rng):
    """-> (N, destination of every group)."""
    if case == "N=1":
        return 1, lambda g: np.zeros_like(g)
    if case == "N=4096, most partitions empty":
        used = rng.choice(4096, 25, replace=False)
        return 4096, lambda g: used[g % len(used)]
    if case == "empty partitions first, middle and last":
        used = np.array([2, 3, 5, 6, 9])
        return 11, lambda g: used[g % len(used)]
    return 16, lambda g: np.full_like(g, 7)  # all rows in one partition


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["N=1", "N=4096, most partitions empty", "empty partitions first, middle and last",
                                  "all rows in one partition"])
def test_partition_layouts(ctx, case):
    rng = np.random.Generator(np.random.PCG64(53))
    N, dest_of = _layout(case, rng)
    n = 20_000
    gid = rng.integers(0, 3000, n)
    ops = [-1, -1, SUM_I64, MAX_F64, SUM_I128]
    cols = [(gid * 977).astype(np.int64), (gid % 3).astype(np.uint16)] + [state_column(op, n, rng) for op in ops[2:]]
    order, starts = by_destination(dest_of(gid), N, rng)
    cols = permuted(cols, order)
    run_and_check(ctx, cols, [0, 1], ops, starts)


@pytest.mark.gpu
def test_same_key_in_two_partitions_is_two_groups(ctx):
    """Groups never cross input partitions, whatever decided the partitions: rows of partition q stay in output partition q."""
    ops = [-1, SUM_I64, MIN_I64]
    cols = [np.array([42, 42], np.int64), np.array([1, 2], np.int64), np.array([5, 6], np.int64)]
    outs, out_starts = reduce_device(ctx, cols, [0], ops, np.array([0, 1, 2], np.int64))
    assert out_starts.tolist() == [0, 1, 2]
    assert outs[1].tolist() == [1, 2] and outs[2].tolist() == [5, 6]
    rng = np.random.Generator(np.random.PCG64(59))
    n, N = 30_000, 6
    key = rng.integers(0, 200, n).astype(np.int64)  # every key in every partition
    ops = [-1] + ALL_OPS
    order, starts = by_destination(rng.integers(0, N, n), N, rng)
    cols = permuted([key] + [state_column(op, n, rng) for op in ALL_OPS], order)
    got = run_and_check(ctx, cols, [0], ops, starts)
    assert len(got) == N * 200


@pytest.mark.gpu
def test_sliced_inputs_honour_the_arrow_offset(ctx):
    """Key and state columns are slices (Arrow offset != 0, a different offset per column) of longer device columns whose
    leading rows hold real keys and all-ones states."""
    rng = np.random.Generator(np.random.PCG64(61))
    n, N = 8_000, 3
    gid = rng.integers(0, 500, n)
    ops = [-1, SUM_I64, -1] + ALL_OPS[1:]
    cols = [(gid % 251).astype(np.uint16), state_column(SUM_I64, n, rng),
            np.stack([gid.astype(np.uint64), (gid * 3).astype(np.uint64)], axis=1)] + [state_column(op, n, rng) for op in ALL_OPS[1:]]
    order, starts = by_destination(gid % N, N, rng)
    cols = permuted(cols, order)
    offsets = [3, 17, 1, 1000, 5, 64, 2, 9, 33]
    run_and_check(ctx, cols, [0, 2], ops, starts, offsets)


@pytest.mark.gpu
def test_argument_errors_leave_the_context_usable(ctx):
    """Every rejected call returns its status; the next valid call on the same context succeeds and is exact."""
    rng = np.random.Generator(np.random.PCG64(67))
    n = 100
    cols = [rng.integers(0, 10, n).astype(np.int64), state_column(SUM_I64, n, rng), state_column(SUM_I128, n, rng)]
    ops = [-1, SUM_I64, SUM_I128]
    starts = np.array([0, 50, n], dtype=np.int64)
    st = Staged(ctx, cols, ops, starts)
    col0, col1 = st.cin[0], st.cin[1]

    def fixed(src, **kw):
        d = nv.DfdColumn(src.kind, src.width, src.values, src.offsets, src.validity, src.offset, src.values_bytes)
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    cases = {  # name -> (in cols, out cols, key cols, ops, n_rows, status)
        "33 columns": (st.cin + [col1] * 30, st.cout + [st.cout[1]] * 30, [0], ops + [SUM_I64] * 30, n, ERR_INVALID_ARGUMENT),
        "9 keys": (st.cin + [col0] * 8, st.cout + [st.cout[0]] * 8, [0] + list(range(3, 11)), ops + [-1] * 8, n, ERR_INVALID_ARGUMENT),
        "3-byte key": ([fixed(col0, width=3)] + st.cin[1:], [fixed(st.cout[0], width=3)] + st.cout[1:], [0], ops, n, ERR_INVALID_ARGUMENT),
        "op 7": (st.cin, st.cout, [0], [-1, 7, SUM_I128], n, ERR_INVALID_ARGUMENT),
        "SUM_I128 on 8 bytes": (st.cin, st.cout, [0], [-1, SUM_I128, SUM_I128], n, ERR_INVALID_ARGUMENT),
        "validity": ([col0, fixed(col1, validity=col1.values), st.cin[2]], st.cout, [0], ops, n, ERR_UNSUPPORTED),
        "var-width key": ([fixed(col0, kind=nv.COL_UTF8, offsets=col1.values, values_bytes=8 * n)] + st.cin[1:], st.cout, [0], ops, n,
                          ERR_UNSUPPORTED),
        "neither key nor aggregate": (st.cin, st.cout, [0], [-1, -1, SUM_I128], n, ERR_INVALID_ARGUMENT),
        "key carries an op": (st.cin, st.cout, [0], [SUM_I64, SUM_I64, SUM_I128], n, ERR_INVALID_ARGUMENT),
        "n_rows = 2^32 - 1": (st.cin, st.cout, [0], ops, (1 << 32) - 1, ERR_INVALID_ARGUMENT),
        "NULL values": ([col0, fixed(col1, values=None), st.cin[2]], st.cout, [0], ops, n, ERR_INVALID_ARGUMENT),
    }
    for name, (cin, cout, keys, o, rows, status) in cases.items():
        host = (C.c_int64 * 3)()
        rc = _call(ctx, cin, rows, keys, o, st.part_starts.ptr, 2, cout, host, st.dev_starts.ptr)
        assert rc == status, (name, rc, nv.lib().dfd_last_error())
        assert nv.check(st.call([0], ops)) is None, name
        check_exact(cols, [0], ops, starts, st.outputs(), st.out_starts)


@pytest.mark.gpu
def test_large_table_beyond_l2(ctx):
    """2^24 rows in 2^23 groups (two rows each) over 16 partitions: the 2^25-slot table and its output-row map (256 MB)
    are far larger than L2.  Checked against the vectorised reference."""
    rng = np.random.Generator(np.random.PCG64(71))
    n, G, N = 1 << 24, 1 << 23, 16
    gid = rng.permutation(np.repeat(np.arange(G, dtype=np.int64), 2))
    key = (gid.astype(np.uint64) * np.uint64(0x9E37_79B9_7F4A_7C15)).view(np.int64)
    ops = [SUM_I64, MIN_I64, MAX_I64, SUM_I128, MIN_F64, MAX_F64]
    vals = [state_column(op, n, rng) for op in ops]
    vals[3][:, 0] |= np.uint64(1 << 63)  # half of the low-limb adds carry
    sb = _special_bits(rng, n)
    vals[4], vals[5] = sb, sb[::-1].copy()
    order, starts = by_destination((gid * 40503) % N, N)
    cols = permuted([key] + vals, order)
    del vals, gid, key, order
    outs, out_starts = reduce_device(ctx, cols, [0], [-1] + ops, starts)
    assert int(out_starts[-1]) == G
    want_p, want_k, want = reduce_reference_np(cols[0], np.repeat(np.arange(N), np.diff(starts)), cols[1:], ops)
    got_p = np.repeat(np.arange(N), np.diff(out_starts))
    o = np.lexsort((outs[0], got_p))
    assert np.array_equal(got_p[o], want_p) and np.array_equal(outs[0][o], want_k)
    for j, op in enumerate(ops):
        g = outs[j + 1][o]
        w = want[j]
        assert np.array_equal(g.view(np.uint64) if op in (MIN_F64, MAX_F64) else g, w), f"op {op}"
