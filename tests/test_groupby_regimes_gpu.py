"""Hash aggregation in each of its three regimes against an exact, vectorised numpy reference.

scan_aggregate (csrc/agg.cu) picks one of three implementations, each with its own accumulators, table and key write-back:
  S  per-CTA shared-memory tables merged into a global table (`aggregate_smem_kernel`): the groups fit the CTA tables;
  G  one global open-addressing table (`aggregate_global_kernel`): S overflowed, or R does not apply;
  R  radix partitioning into TMA-fed shared-memory tables (`radix_agg_kernel`): more than 2^20 rows, the 256 K-row
     cardinality probe overflows, fixed-width NOT NULL keys of at most 16 bytes, no float aggregate, at most 5 value
     columns, and a shared-memory budget that leaves at least 1024 table slots (radix_groupby).
Every GPU test asserts from the profiler's kernel records which regime ran: a spec list over R's budget silently falls back
to G, so a test that does not check would stop covering R without failing.  High-cardinality inputs run through R and,
with B2_AGG_NO_RADIX set, through G; both must equal the reference and each other.

`reference_groupby` groups on normalised key bits (NULL is its own group, -0.0 == 0.0, all NaNs are one group) by a sort
and numpy reduceat, with no loop over rows.  INT64 sums wrap mod 2^64 like Spark's non-ANSI long sum; decimal sums are
exact, summed in 32-bit limbs and NULL when they need more than the result precision.  test_reference_matches_oracle pins
it to oracle.spark_cpu on a few thousand rows from the same generators, without a GPU."""
import numpy as np
import pytest

from oracle import spark_cpu as O

N_BIG = 1_200_000                 # > 2^20 rows: the cardinality probe runs and R is possible
M32 = np.uint64(0xFFFFFFFF)
RADIX, GLOBAL, SMEM = "radix_agg_kernel", "aggregate_global_kernel", "aggregate_smem_kernel"
I64_MIN, I64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max


class Col:
    """values (DECIMAL128: (n, 2) uint64 low/high words of the two's-complement value), valid, typ = (dtype, precision, scale)"""

    def __init__(self, values, typ, valid=None):
        self.values = values
        self.typ = typ
        self.valid = np.ones(len(values), bool) if valid is None else np.asarray(valid, bool)

    @property
    def nullable(self):
        return not self.valid.all()

    def take(self, idx):
        return Col(self.values[idx], self.typ, self.valid[idx])


def d128_words(ints):
    """python ints -> (n, 2) uint64 words"""
    return np.array([(v & (2**64 - 1), (v >> 64) & (2**64 - 1)) for v in ints], dtype=np.uint64).reshape(-1, 2)


def d128_ints(words):
    """(n, 2) uint64 words -> object array of python ints"""
    return words[:, 1].view(np.int64).astype(object) * (1 << 64) + words[:, 0].astype(object)


def to_ocol(c):
    dt = c.typ[0]
    if dt == O.DECIMAL128:
        return O.OCol(d128_ints(c.values), c.valid, c.typ)
    if O.is_decimal(dt):
        return O.OCol(c.values.astype(np.int64).astype(object), c.valid, c.typ)
    return O.OCol(c.values, c.valid, c.typ)


# ------------------------------------------------------------------------------------------------------------------------------
# the reference
def key_bits(values, valid, normalise):
    """int64 grouping bits per row, 0 under NULL; floats as their bit pattern, normalised (+0.0, canonical NaN) on request"""
    v = values
    if v.dtype == np.float32:
        if normalise:
            with np.errstate(invalid="ignore"):      # signalling NaN payloads
                v = np.where(np.isnan(v), np.float32(np.nan), v + np.float32(0.0))
        b = np.ascontiguousarray(v).view(np.uint32).astype(np.int64)
    elif v.dtype == np.float64:
        if normalise:
            with np.errstate(invalid="ignore"):
                v = np.where(np.isnan(v), np.nan, v + 0.0)
        b = np.ascontiguousarray(v).view(np.int64)
    else:
        b = v.astype(np.int64)
    return np.where(valid, b, 0)


def key_matrix(keys, normalise):
    """(n, 2 * nkeys) int64: (valid, bits) of every key"""
    n = len(keys[0][0])
    m = np.zeros((n, 2 * len(keys)), np.int64)
    for i, (v, ok) in enumerate(keys):
        m[:, 2 * i] = ok
        m[:, 2 * i + 1] = key_bits(v, ok, normalise)
    return m


def _words(c):
    """(low 64 bits as uint64, high 64 bits as int64) of every value of an integral or decimal column"""
    if c.typ[0] == O.DECIMAL128:
        return np.ascontiguousarray(c.values[:, 0]), np.ascontiguousarray(c.values[:, 1]).view(np.int64)
    v = c.values.astype(np.int64)
    return v.view(np.uint64), v >> 63


def reference_groupby(keys, cols, specs, nrows):
    """keys: list of Col; cols: the columns specs refer to.  -> (key matrix of the groups in lexicographic order,
    [(values, valid)] per spec).  No keys: one group, also over zero rows."""
    if keys:
        m = key_matrix([(k.values, k.valid) for k in keys], True)
        order = np.lexsort(m.T[::-1])
        ms = m[order]
        starts = np.flatnonzero(np.r_[True, (ms[1:] != ms[:-1]).any(axis=1)]) if nrows else np.zeros(0, np.int64)
        kmat = ms[starts]
    else:
        order, starts, kmat = np.arange(nrows), np.zeros(1, np.int64), np.zeros((1, 0), np.int64)
    ng = len(starts)

    def red(ufunc, x):
        return ufunc.reduceat(x[order], starts) if nrows and ng else np.zeros(ng, x.dtype)

    out = []
    for spec in specs:
        kind = spec[0]
        if kind == O.AGG_COUNT_ALL:
            out.append((np.diff(np.r_[starts, nrows]).astype(np.int64), np.ones(ng, bool)))
            continue
        c = cols[spec[1]]
        cnt = red(np.add, c.valid.astype(np.int64))
        if kind == O.AGG_COUNT:
            out.append((cnt, np.ones(ng, bool)))
            continue
        has = cnt > 0
        if kind in (O.AGG_MIN, O.AGG_MAX):
            fill = I64_MAX if kind == O.AGG_MIN else I64_MIN
            out.append((red(np.minimum if kind == O.AGG_MIN else np.maximum, np.where(c.valid, c.values.astype(np.int64), fill)), has))
        elif c.typ[0] in (O.FLOAT32, O.FLOAT64):
            # integer-valued test data: every partial sum is exact in float64, whatever the order
            out.append((red(np.add, np.where(c.valid, c.values.astype(np.float64), 0.0)), has))
        elif not O.is_decimal(c.typ[0]):
            out.append((red(np.add, np.where(c.valid, c.values.astype(np.int64), 0)), has))   # int64 reduceat wraps mod 2^64
        else:
            # exact: 32-bit limbs (three unsigned, the top one signed) summed per group in int64 (exact below 2^31 rows a
            # group), recombined as python ints
            lo, hi = _words(c)
            lo, hi = np.where(c.valid, lo, np.uint64(0)), np.where(c.valid, hi, 0)
            limbs = [(lo & M32).astype(np.int64), (lo >> np.uint64(32)).astype(np.int64), (hi.view(np.uint64) & M32).astype(np.int64), hi >> 32]
            s = sum(red(np.add, l).astype(object) * (1 << (32 * i)) for i, l in enumerate(limbs))
            fits = np.array([abs(x) < 10 ** spec[4] for x in s], dtype=bool) if ng else np.zeros(0, bool)
            out.append((s, has & fits))
    return kmat, out


# ------------------------------------------------------------------------------------------------------------------------------
# running on the GPU
def kernels_run(b2, fn):
    """-> (fn(), {kernel name: launches}) for this call alone (profile_enable clears earlier records)"""
    b2.profile_enable(True)
    try:
        out = fn()
        ran = {r["name"]: r["launches"] for r in b2.profile_report()}
    finally:
        b2.profile_enable(False)
    return out, ran


def regimes(ran):
    return {k for k in (SMEM, GLOBAL, RADIX) if k in ran}


def to_b2(b2, c):
    return b2.Column.from_numpy(c.values, dtype=c.typ[0], valid=c.valid if c.nullable else None, scale=c.typ[2])


def read_col(b2, col):
    """-> (values, valid); DECIMAL128 as python ints, read as raw words (no per-row conversion in the library wrapper)"""
    if col.dtype == b2.DECIMAL128:
        from spark_rapids_b200 import _init as I
        n = len(col)
        words = np.zeros((n, 2), np.uint64)
        vb = np.zeros((n + 7) // 8, np.uint8)
        I.check(I.lib.b2_column_to_host(col.h, I._ptr(words), I._ptr(vb), None))
        return d128_ints(words), I.unpack_bits(vb, n)
    return col.to_numpy()


def canonical(keys, aggs):
    """result columns in the order of their key matrix (raw key bits: a -0.0 or NaN payload in the output stays visible)"""
    m = key_matrix(keys, False) if keys else np.zeros((len(aggs[0][0]), 0), np.int64)
    order = np.lexsort(m.T[::-1]) if keys else np.arange(len(m))
    return m[order], [(v[order], ok[order]) for v, ok in aggs]


def assert_result(got, exp):
    (gm, gaggs), (em, eaggs) = got, exp
    assert gm.shape == em.shape, "groups: got %d, expected %d" % (len(gm), len(em))
    bad = np.flatnonzero((gm != em).any(axis=1)) if len(gm) else []
    assert len(bad) == 0, "%d key rows differ, first got %s expected %s" % (len(bad), gm[bad[0]], em[bad[0]])
    for k, ((gv, gok), (ev, eok)) in enumerate(zip(gaggs, eaggs)):
        assert np.array_equal(gok, eok), "aggregate %d: validity differs in %d groups" % (k, int((gok != eok).sum()))
        diff = np.flatnonzero(gok & (gv != ev))
        assert len(diff) == 0, "aggregate %d: %d values differ, first got %r expected %r" % (k, len(diff), gv[diff[0]], ev[diff[0]])


def aggregate(b2, table, cols, key_idx, specs, pred=None):
    """scan_aggregate over a program that passes every column through (plus an optional fused predicate as output 0), so
    that aggregates over the same column share one program output -> (result table, kernels run)"""
    outs = [b2.col(i, c.typ[0], c.typ[1], c.typ[2], nullable=c.nullable) for i, c in enumerate(cols)]
    prog = b2.Program(([pred(outs)] if pred else []) + outs)
    return kernels_run(b2, lambda: b2.scan_aggregate(prog, pred is not None, table, key_idx, specs))


def check_regime(b2, table, cols, key_idx, specs, expect, want, pred=None, key_of=None):
    """run, assert the regimes that ran, compare with the reference result `want`; -> the canonical result"""
    out, ran = aggregate(b2, table, cols, key_idx, specs, pred)
    assert regimes(ran) == expect, ran
    res = [read_col(b2, out.column(i)) for i in range(out.num_columns)]
    keys = [(key_of(v) if key_of else v, ok) for v, ok in res[:len(key_idx)]]
    got = canonical(keys, res[len(key_idx):])
    assert_result(got, want)
    return got, ran


def check_r_and_g(b2, monkeypatch, cols, key_idx, specs, pred_np=None, pred=None, key_of=None):
    """the same input through R and through G: both equal the reference, and each other"""
    table = b2.Table.from_columns([to_b2(b2, c) for c in cols])
    sel = cols if pred_np is None else [c.take(pred_np) for c in cols]
    want = reference_groupby([sel[k] for k in key_idx], sel, specs, len(sel[0].values))
    r, _ = check_regime(b2, table, cols, key_idx, specs, {RADIX}, want, pred, key_of)
    monkeypatch.setenv("B2_AGG_NO_RADIX", "1")
    g, _ = check_regime(b2, table, cols, key_idx, specs, {GLOBAL}, want, pred, key_of)
    monkeypatch.delenv("B2_AGG_NO_RADIX")
    assert_result(r, g)


# ------------------------------------------------------------------------------------------------------------------------------
# data
D128 = (O.DECIMAL128, 38, 2)
D64 = (O.DECIMAL64, 18, 0)
D32 = (O.DECIMAL32, 9, 2)
BIG128 = 10**38 - 1


def edge_columns(seed, ngroups, per_group):
    """value edges, `per_group` rows in each of `ngroups` groups, rows shuffled.  Group type g % 4 sets the signs of the
    near-limit values: 0 all positive (sums pass 2^127 / 2^63 / the result precision), 2 all negative, 1 alternating (sums
    come back into range), 3 alternating with one more positive row (ends just out of range).
      0 key INT64 (negative and positive)   1 INT64 ~ +-2^62       2 DECIMAL128(38,2) ~ +-(10^38-1)
      3 DECIMAL64(18,0) ~ +-(10^18-1)       4 DECIMAL32(9,2)        5 INT8   6 INT16   7 INT32 (full range)
      8 INT64 ~ +-2^62, nullable (groups g % 5 == 0 all NULL)       9 DECIMAL128, nullable (groups g % 7 == 0 all NULL)"""
    rng = np.random.default_rng(seed)
    n = ngroups * per_group
    perm = rng.permutation(n)
    g, j = np.repeat(np.arange(ngroups), per_group)[perm], np.tile(np.arange(per_group), ngroups)[perm]
    t = g % 4
    sign = np.where(t == 0, 1, np.where(t == 2, -1, np.where((j % 2 == 0) | ((t == 3) & (j == 1)), 1, -1))).astype(np.int64)
    small = rng.integers(0, 1000, n)
    mags = d128_words([s * (BIG128 - d) for s in (1, -1) for d in range(1000)])
    d128 = mags[np.where(sign > 0, 0, 1000) + small]
    cols = [Col((g * 7919 - ngroups * 3000).astype(np.int64), (O.INT64, 0, 0)),
            Col(sign * (2**62 - small), (O.INT64, 0, 0)),
            Col(d128, D128),
            Col(sign * (10**18 - 1 - small), D64),
            Col((sign * (10**9 - 1 - small)).astype(np.int32), D32),
            Col(rng.integers(-128, 128, n).astype(np.int8), (O.INT8, 0, 0)),
            Col(rng.integers(-2**15, 2**15, n).astype(np.int16), (O.INT16, 0, 0)),
            Col(rng.integers(-2**31, 2**31, n).astype(np.int32), (O.INT32, 0, 0)),
            Col(-sign * (2**62 - small), (O.INT64, 0, 0), (g % 5 != 0) & (rng.random(n) > 0.3)),
            Col(mags[np.where(sign > 0, 1000, 0) + small[::-1]], D128, (g % 7 != 0) & (rng.random(n) > 0.3))]
    return cols


# spec lists over edge_columns, each inside R's budget (<= 5 value columns, >= 1024 table slots); one program output per
# column, so the aggregates of one column share a value slot
EDGE_SPECS = {
    "int64_and_decimal128_sums": [(O.AGG_SUM, 1, O.INT64, 0, 0), (O.AGG_SUM, 2, O.DECIMAL128, 2, 38), (O.AGG_COUNT_ALL, 0), (O.AGG_COUNT, 1)],
    "narrow_decimal_sums": [(O.AGG_SUM, 3, O.DECIMAL64, 0, 18), (O.AGG_SUM, 3, O.DECIMAL128, 0, 38), (O.AGG_MIN, 3), (O.AGG_MAX, 3),
                            (O.AGG_SUM, 4, O.DECIMAL64, 2, 10)],
    "min_max": [(O.AGG_MIN, 5), (O.AGG_MAX, 5), (O.AGG_MIN, 6), (O.AGG_MAX, 6), (O.AGG_MIN, 7), (O.AGG_MAX, 7), (O.AGG_MIN, 1), (O.AGG_MAX, 1)],
    "nullable_values": [(O.AGG_SUM, 8, O.INT64, 0, 0), (O.AGG_COUNT, 8), (O.AGG_COUNT_ALL, 0), (O.AGG_MIN, 8), (O.AGG_MAX, 8),
                        (O.AGG_SUM, 9, O.DECIMAL128, 2, 38), (O.AGG_COUNT, 9)],
}


def float_key_values(dtype, n, rng, nrandom):
    """keys with -0.0 and no +0.0 (the zero group is made only of -0.0), NaNs with non-canonical payloads only, infinities,
    and `nrandom` other integral values"""
    if dtype == np.float64:
        nans = np.array([0x7FF8000000000001, 0xFFF8000000000000, 0x7FF0000000000001, 0x7FFFFFFFFFFFFFFF], np.uint64).view(np.float64)
    else:
        nans = np.array([0x7FC00001, 0xFFC00000, 0x7F800001, 0x7FFFFFFF], np.uint32).view(np.float32)
    special = np.concatenate([nans, np.array([-0.0, np.inf, -np.inf], dtype)])
    pool = np.concatenate([special, (rng.permutation(4 * nrandom)[:nrandom] - 2 * nrandom).astype(dtype)])
    pool[len(special):][pool[len(special):] == 0] = 1.5                      # no +0.0: zero only ever appears as -0.0
    pick = rng.integers(0, len(pool), n)
    pick[:len(special)] = np.arange(len(special))                             # every special value is present
    return pool[pick]


def key_shape_columns(shape, n, ngroups, seed):
    """key columns of one shape, drawn from a pool of `ngroups` key tuples, then an INT64 value column"""
    rng = np.random.default_rng(seed)
    pick = rng.integers(0, ngroups, n)

    def full(dt, lo, hi):
        v = rng.integers(lo, hi, ngroups, endpoint=True, dtype=np.int64)
        v[:4] = [lo, hi, -1, 0]
        return v.astype(dt)[pick]

    i64 = lambda: full(np.int64, I64_MIN, I64_MAX)
    if shape == "int64":
        keys = [Col(i64(), (O.INT64, 0, 0))]
    elif shape == "date32_int8_int32_int16":          # 11 bytes: k0 and k1, the DATE32 at bit 0, INT32 across the two words
        keys = [Col(full(np.int32, -25567, 47482), (O.DATE32, 0, 0)), Col(full(np.int8, -128, 127), (O.INT8, 0, 0)),
                Col(full(np.int32, -2**31, 2**31 - 1), (O.INT32, 0, 0)), Col(full(np.int16, -2**15, 2**15 - 1), (O.INT16, 0, 0))]
    elif shape == "int32_int8_int16":                 # 7 bytes: packed fast keys in S and G, k0 only in R
        keys = [Col(full(np.int32, -2**31, 2**31 - 1), (O.INT32, 0, 0)), Col(full(np.int8, -128, 127), (O.INT8, 0, 0)),
                Col(full(np.int16, -2**15, 2**15 - 1), (O.INT16, 0, 0))]
    elif shape == "int64_int64":
        keys = [Col(i64(), (O.INT64, 0, 0)), Col(i64(), (O.INT64, 0, 0))]
    elif shape == "decimal64":
        keys = [Col(full(np.int64, -(10**18 - 1), 10**18 - 1), D64)]
    elif shape in ("float64", "float32"):
        dt = np.float64 if shape == "float64" else np.float32
        keys = [Col(float_key_values(dt, n, rng, ngroups), (O.FLOAT64 if dt == np.float64 else O.FLOAT32, 0, 0))]
    else:
        raise ValueError(shape)
    return keys + [Col(rng.integers(-2**62, 2**62, n), (O.INT64, 0, 0))]


# ------------------------------------------------------------------------------------------------------------------------------
# the reference against the oracle (no GPU)
def _rows(kmat, aggs):
    """sorted python rows: key (valid, bits) pairs, then every aggregate as None / int / float"""
    def py(v):
        return float(v) if isinstance(v, (float, np.floating)) else int(v)
    cols = [[py(v) if ok else None for v, ok in zip(vals, valid)] for vals, valid in aggs]
    keys = [tuple(int(x) for x in r) for r in kmat]
    return sorted(zip(keys, *cols), key=repr)


def _oracle_rows(ocols, nkeys):
    keys = key_matrix([(c.values, c.valid) for c in ocols[:nkeys]], False) if nkeys else np.zeros((len(ocols[0]), 0), np.int64)
    aggs = [(np.array(c.to_pylist(), dtype=object), c.valid) for c in ocols[nkeys:]]
    return _rows(keys, [(np.where(ok, v, 0), ok) for v, ok in aggs])


def _small_cases():
    rng = np.random.default_rng(5)
    edge = edge_columns(3, 250, 12)
    for name, specs in EDGE_SPECS.items():
        yield "edge/" + name, edge, [0], specs
        yield "edge_reduce/" + name, edge, [], specs
        yield "edge_reduce_empty/" + name, [c.take(slice(0, 0)) for c in edge], [], specs
    for shape in ("int64", "date32_int8_int32_int16", "int32_int8_int16", "int64_int64", "decimal64", "float64", "float32"):
        cols = key_shape_columns(shape, 3000, 1000, 7)
        nk = len(cols) - 1
        yield "keys/" + shape, cols, list(range(nk)), [(O.AGG_SUM, nk, O.INT64, 0, 0), (O.AGG_COUNT_ALL, 0), (O.AGG_MAX, nk)]
    k = key_shape_columns("int64", 3000, 500, 8)
    k[0].valid = rng.random(3000) > 0.1
    fsum = Col(rng.integers(-1000, 1000, 3000).astype(np.float64), (O.FLOAT64, 0, 0), rng.random(3000) > 0.2)
    yield "nullable_key_float_sum", k + [fsum], [0], [(O.AGG_SUM, 2, O.FLOAT64, 0, 0), (O.AGG_COUNT, 2), (O.AGG_SUM, 1, O.INT64, 0, 0)]


def test_reference_matches_oracle():
    """the vectorised reference equals oracle.spark_cpu (row-at-a-time python) on every edge the GPU cases use: wrapped
    INT64 sums, DECIMAL128 sums past 2^127 and back, decimal overflow to NULL, narrow decimals, negative MIN/MAX, all-NULL
    groups, NULL keys, -0.0 / NaN payload keys (normalised in the output), empty reductions"""
    for name, cols, key_idx, specs in _small_cases():
        n = len(cols[0].values)
        ocols = [to_ocol(c) for c in cols]
        want = O.groupby_cols(ocols, key_idx, specs) if key_idx else O.reduce_cols(ocols, specs)
        got = reference_groupby([cols[k] for k in key_idx], cols, specs, n)
        assert _rows(*got) == _oracle_rows(want, len(key_idx)), name


# ------------------------------------------------------------------------------------------------------------------------------
# GPU cases
_DATA = {}


def cached(name, make):
    if name not in _DATA:
        _DATA[name] = make()
    return _DATA[name]


@pytest.mark.gpu
@pytest.mark.parametrize("specs", list(EDGE_SPECS), ids=list(EDGE_SPECS))
def test_value_edges_radix_and_global(b2, monkeypatch, specs):
    """100 K groups of 12 rows: wrapping INT64 sums, DECIMAL128 sums past 2^127 (third limb) that end in range or NULL,
    DECIMAL64 -> DECIMAL64(18) overflowing its two limbs to NULL, DECIMAL32, MIN/MAX over negative narrow ints, NULL values
    with all-NULL groups, COUNT(col) next to COUNT(*)"""
    cols = cached("edge_big", lambda: edge_columns(1, 100_000, 12))
    check_r_and_g(b2, monkeypatch, cols, [0], EDGE_SPECS[specs])


@pytest.mark.gpu
@pytest.mark.parametrize("specs", list(EDGE_SPECS), ids=list(EDGE_SPECS))
def test_value_edges_smem(b2, specs):
    """the same value edges in the shared-memory regime: 64 groups over 1.2 M rows (the widest spec list leaves a CTA table
    of 128 slots, abandoned at 7/8 full, so a few hundred groups would overflow into G)"""
    cols = cached("edge_smem", lambda: edge_columns(2, 64, 18_750))
    specs = EDGE_SPECS[specs]
    table = b2.Table.from_columns([to_b2(b2, c) for c in cols])
    check_regime(b2, table, cols, [0], specs, {SMEM}, reference_groupby([cols[0]], cols, specs, len(cols[0].values)))


KEY_SHAPES = ["int64", "date32_int8_int32_int16", "int32_int8_int16", "int64_int64", "decimal64", "float64", "float32"]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", KEY_SHAPES)
def test_key_shapes_radix_and_global(b2, monkeypatch, shape):
    """~300 K groups over 1.2 M rows per key shape: full-range INT64 (one key word), negative narrow keys packed next to each
    other (a sign bit must not leak into the neighbouring key, in R's 128-bit key and in the packed fast keys of G),
    16-byte keys, a DECIMAL64 key, float keys with -0.0 and NaN payloads (output keys are +0.0 and the canonical NaN)"""
    cols = key_shape_columns(shape, N_BIG, 300_000, 11)
    nk = len(cols) - 1
    check_r_and_g(b2, monkeypatch, cols, list(range(nk)), [(O.AGG_SUM, nk, O.INT64, 0, 0), (O.AGG_COUNT_ALL, 0), (O.AGG_MAX, nk)])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["float64", "float32"])
@pytest.mark.parametrize("n", [3000, N_BIG])
def test_float_keys_normalised_smem(b2, dtype, n):
    """few groups, so the shared-memory regime: the zero group holds only -0.0 rows and the NaN group only non-canonical
    payloads, yet the output keys must be +0.0 and the canonical NaN whichever row represents the group"""
    rng = np.random.default_rng(13)
    cols = [Col(float_key_values(dtype, n, rng, 40), (O.FLOAT64 if dtype == np.float64 else O.FLOAT32, 0, 0)),
            Col(rng.integers(-2**62, 2**62, n), (O.INT64, 0, 0))]
    specs = [(O.AGG_SUM, 1, O.INT64, 0, 0), (O.AGG_COUNT_ALL, 0)]
    table = b2.Table.from_columns([to_b2(b2, c) for c in cols])
    (keys, _), _ = check_regime(b2, table, cols, [0], specs, {SMEM}, reference_groupby([cols[0]], cols, specs, n))
    canon = 0x7FF8000000000000 if dtype == np.float64 else 0x7FC00000
    assert 0 in keys[:, 1] and canon in keys[:, 1]


def q3_columns(n, ngroups, seed):
    """l_orderkey INT64, o_orderdate DATE32 (a function of the order key), o_shippriority INT32, l_extendedprice and
    l_discount DECIMAL64(12, 2), l_shipdate DATE32, row id INT32"""
    rng = np.random.default_rng(seed)
    ok = rng.permutation(4 * ngroups)[:ngroups].astype(np.int64)[rng.integers(0, ngroups, n)]
    return [Col(ok, (O.INT64, 0, 0)), Col((ok % 2406 + 8036).astype(np.int32), (O.DATE32, 0, 0)), Col(np.zeros(n, np.int32), (O.INT32, 0, 0)),
            Col(rng.integers(90000, 10494951, n), (O.DECIMAL64, 12, 2)), Col(rng.integers(0, 11, n), (O.DECIMAL64, 12, 2)),
            Col(rng.integers(8036, 10561, n).astype(np.int32), (O.DATE32, 0, 0)), Col(np.arange(n, dtype=np.int32), (O.INT32, 0, 0))]


def run_q3(b2, cols, pred, keep):
    """fused predicate + computed DECIMAL128 value price * (1 - disc) grouped by (orderkey, orderdate, shippriority)"""
    c = [b2.col(i, x.typ[0], x.typ[1], x.typ[2], nullable=False) for i, x in enumerate(cols)]
    rev = c[3] * (b2.lit(1, b2.DECIMAL32, 1, 0) - c[4])
    prog = b2.Program([pred(c), c[0], c[1], c[2], rev])
    assert rev.type()[0] == b2.DECIMAL128 and rev.type()[2] == 4
    # the numpy value is the oracle's on a prefix
    pre = [to_ocol(x.take(slice(0, 2000))) for x in cols]
    assert list(O.eval_expr(rev.sexpr, pre).values) == list(cols[3].values[:2000] * (100 - cols[4].values[:2000]))
    val = cols[3].values * (100 - cols[4].values)
    sel = [cols[0].take(keep), cols[1].take(keep), cols[2].take(keep), Col(val[keep], (O.DECIMAL64, 18, 4))]   # |value| < 2^63
    specs = [(O.AGG_SUM, 3, O.DECIMAL128, 4, 36), (O.AGG_COUNT_ALL, 0)]
    table = b2.Table.from_columns([to_b2(b2, x) for x in cols])
    out, ran = kernels_run(b2, lambda: b2.scan_aggregate(prog, True, table, [0, 1, 2], specs))
    res = [read_col(b2, out.column(i)) for i in range(out.num_columns)]
    assert_result(canonical(res[:3], res[3:]), reference_groupby(sel[:3], sel, specs, int(keep.sum())))
    return ran


@pytest.mark.gpu
def test_q3_shape_radix_predicate_compaction(b2):
    """3 M rows, about half pass the fused predicate (~0.8 M groups among them): R compacts the surviving rows, and ~1.5 M
    rows need P = 2048 partitions, i.e. two 8-bit-or-less scatter passes.  A predicate that keeps only the first 150 K rows,
    each its own group, still overflows the 256 K-row probe, and P = 256 needs one pass."""
    n = 3_000_000
    cols = q3_columns(n, 1_000_000, 17)
    ran = run_q3(b2, cols, lambda c: c[5] > b2.lit(9298, b2.DATE32), cols[5].values > 9298)
    assert regimes(ran) == {RADIX}, ran
    assert ran.get("part_scatter2_kernel", 0) + ran.get("part_scatter_kernel", 0) == 2, ran
    cols[0].values[:150_000] = np.arange(150_000) * 3 + 7
    cols[1].values[:150_000] = (cols[0].values[:150_000] % 2406 + 8036).astype(np.int32)
    ran = run_q3(b2, cols, lambda c: c[6] < b2.lit(150_000, b2.INT32), cols[6].values < 150_000)
    assert regimes(ran) == {RADIX}, ran
    assert ran.get("part_scatter2_kernel", 0) + ran.get("part_scatter_kernel", 0) == 1, ran


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["over_radix_smem_budget", "six_value_columns"])
def test_wide_spec_lists_fall_back_to_global(b2, case):
    """a DECIMAL128 sum, two narrow decimal sums and MIN/MAX of two columns on two INT64 keys leave fewer than 1024 slots in
    R's shared memory; six value columns exceed R's five.  Both must end in G with the exact result."""
    cols = cached("edge_big", lambda: edge_columns(1, 100_000, 12))
    cols = cols + [Col(cols[0].values * 3 + 1, (O.INT64, 0, 0))]
    if case == "over_radix_smem_budget":
        keys, specs = [0, 10], [(O.AGG_SUM, 2, O.DECIMAL128, 2, 38), (O.AGG_SUM, 3, O.DECIMAL128, 0, 38), (O.AGG_SUM, 4, O.DECIMAL64, 2, 18),
                                (O.AGG_MIN, 7), (O.AGG_MAX, 7), (O.AGG_MIN, 1), (O.AGG_MAX, 1)]
    else:
        keys, specs = [0], [(O.AGG_SUM, 1, O.INT64, 0, 0), (O.AGG_SUM, 2, O.DECIMAL128, 2, 38), (O.AGG_SUM, 3, O.DECIMAL64, 0, 18),
                            (O.AGG_SUM, 4, O.DECIMAL64, 2, 18), (O.AGG_MIN, 5), (O.AGG_MAX, 6)]
    table = b2.Table.from_columns([to_b2(b2, c) for c in cols])
    check_regime(b2, table, cols, keys, specs, {GLOBAL}, reference_groupby([cols[k] for k in keys], cols, specs, len(cols[0].values)))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["nullable_key", "string_key", "float_sum"])
def test_inputs_radix_cannot_take_fall_back_to_global(b2, case):
    """~300 K groups over 1.2 M rows (the probe overflows) with a nullable key, a STRING key or a float SUM: R does not apply"""
    rng = np.random.default_rng(19)
    cols = key_shape_columns("int64", N_BIG, 300_000, 19)
    specs = [(O.AGG_SUM, 1, O.INT64, 0, 0), (O.AGG_COUNT_ALL, 0)]
    key_of = None
    if case == "nullable_key":
        cols[0].valid = rng.random(N_BIG) > 0.05
    elif case == "float_sum":
        cols.append(Col(rng.integers(-1000, 1000, N_BIG).astype(np.float64), (O.FLOAT64, 0, 0)))
        specs.append((O.AGG_SUM, 2, O.FLOAT64, 0, 0))
    if case == "string_key":
        ids = rng.integers(0, 300_000, N_BIG) * 31 + 10_000_000                  # 8 decimal digits
        chars = ((ids[:, None] // 10 ** np.arange(7, -1, -1)) % 10 + 48).astype(np.uint8).ravel()
        scol = b2.Column.from_string_buffers(chars, np.arange(N_BIG + 1, dtype=np.int32) * 8)
        cols[0] = Col(ids, (O.STRING, 0, 0))
        table = b2.Table.from_columns([scol, to_b2(b2, cols[1])])
        key_of = lambda v: np.array([int(x) for x in v], np.int64)    # noqa: E731
    else:
        table = b2.Table.from_columns([to_b2(b2, c) for c in cols])
    check_regime(b2, table, cols, [0], specs, {GLOBAL}, reference_groupby([cols[0]], cols, specs, N_BIG), key_of=key_of)


@pytest.mark.gpu
def test_probe_passes_then_smem_overflows_into_global(b2):
    """keys sorted so that the 256 K-row probe sees 27 groups and the rest of the input ~300 K: the probe passes, the
    shared-memory tables overflow, and the call ends in G with the exact result"""
    rng = np.random.default_rng(23)
    key = np.concatenate([np.arange(300_000) // 10_000, rng.integers(1000, 301_000, N_BIG - 300_000)]).astype(np.int64)
    cols = [Col(key, (O.INT64, 0, 0)), Col(rng.integers(-2**62, 2**62, N_BIG), (O.INT64, 0, 0))]
    specs = [(O.AGG_SUM, 1, O.INT64, 0, 0), (O.AGG_COUNT_ALL, 0), (O.AGG_MIN, 1)]
    table = b2.Table.from_columns([to_b2(b2, c) for c in cols])
    check_regime(b2, table, cols, [0], specs, {SMEM, GLOBAL}, reference_groupby([cols[0]], cols, specs, N_BIG))


@pytest.mark.gpu
@pytest.mark.parametrize("keyed", [True, False], ids=["keyed", "keyless"])
def test_predicate_keeps_nothing(b2, keyed):
    """1.2 M rows, none pass: keyed -> no rows; keyless -> one row, NULL sums and zero counts.  Nothing passes in the probe
    either, so this is S (R's own m == 0 return needs a probe that overflowed, i.e. surviving rows)."""
    rng = np.random.default_rng(29)
    cols = [Col(rng.integers(0, 300_000, N_BIG), (O.INT64, 0, 0)), Col(rng.integers(-2**62, 2**62, N_BIG), (O.INT64, 0, 0)),
            Col(d128_words([10**37])[np.zeros(N_BIG, np.int64)], D128), Col(np.arange(N_BIG, dtype=np.int32), (O.INT32, 0, 0))]
    specs = [(O.AGG_SUM, 1, O.INT64, 0, 0), (O.AGG_SUM, 2, O.DECIMAL128, 2, 38), (O.AGG_COUNT, 1), (O.AGG_COUNT_ALL, 0), (O.AGG_MAX, 1)]
    keys = [0] if keyed else []
    table = b2.Table.from_columns([to_b2(b2, c) for c in cols])
    none = [c.take(slice(0, 0)) for c in cols]
    got, _ = check_regime(b2, table, cols, keys, specs, {SMEM}, reference_groupby([none[k] for k in keys], none, specs, 0),
                          pred=lambda c: c[3] < b2.lit(0, b2.INT32))
    assert len(got[1][0][0]) == (0 if keyed else 1)


@pytest.mark.gpu
def test_exec_partial_merge_runs_in_radix(b2):
    """GpuHashAggregateExec (partial) over 3 batches of 600 K rows: each batch's partial has ~420 K groups, so the merge
    pass over the concatenated partials (> 2^20 rows) runs in R.  The merged DECIMAL128 sum of sums and the counts merged
    as INT64 sums equal a one-pass aggregation of all rows."""
    from spark_rapids_b200 import execs as E
    rng = np.random.default_rng(31)
    per, nb = 600_000, 3
    n = per * nb
    pool = d128_words([(-1) ** i * (10**30 + i * 12345678901234567) for i in range(2000)])
    cols = [Col(rng.integers(0, 800_000, n), (O.INT64, 0, 0)), Col(pool[rng.integers(0, 2000, n)], D128)]
    batches = [b2.Table.from_columns([to_b2(b2, c.take(slice(i * per, (i + 1) * per))) for c in cols]) for i in range(nb)]
    pre = [b2.col(0, b2.INT64, nullable=False), b2.col(1, b2.DECIMAL128, 38, 2, nullable=False)]
    specs = [(O.AGG_SUM, 1, O.DECIMAL128, 2, 38), (O.AGG_COUNT_ALL, 0), (O.AGG_COUNT, 1)]
    agg = E.GpuHashAggregateExec(E.GpuBatchSource(batches), [0], specs, pre_project=pre)
    out, ran = kernels_run(b2, agg.collect)
    assert ran.get(RADIX) == 1, ran
    res = [read_col(b2, out.column(i)) for i in range(out.num_columns)]
    assert_result(canonical(res[:1], res[1:]), reference_groupby([cols[0]], cols, specs, n))
