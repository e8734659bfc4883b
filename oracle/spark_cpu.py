"""oracle/spark_cpu.py — CPU restatement of the Spark/RAPIDS semantics of the hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under spark-rapids_b200/ may import this; it is the checker used
by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs.

The reference's arithmetic lives in an un-vendored dependency (com.nvidia:spark-rapids-jni
26.06.0-SNAPSHOT, classifier cuda12: cudf-java/libcudf; pom.xml:834-836, 1036-1041) and cannot be
built or run here (no JVM/Spark/cudf).  This file therefore restates the *Spark semantics* that the
reference's Scala call sites document and that its differential tests enforce (CPU Spark == GPU):

  expressions  sql-plugin/.../rapids/predicates.scala:54-331, arithmetic.scala:38-126, 309-340,
               411-640, GpuCast.scala:295, conditionalExpressions.scala, nullExpressions.scala
  filter       basicPhysicalOperators.scala:1148-1224
  aggregates   GpuAggregateExec.scala:540-585, aggregate/aggregateFunctions.scala:38-68, 1041-1290,
               1408-1683
  (hash, join, sort, parquet, rows live in the sibling modules)

PINNING: the reference holds almost no golden vectors for this path (SURVEY.md §8c).  Pinned by
tests/test_oracle_golden.py against: HashAggregateRetrySuite.scala:34-52,117-206 (sum{5,null,3,1}=9;
group-by {5->1,null->2,1->7}), Spark Murmur3 known answers, GpuPartitioningSuite.scala:112-225
slice counts, and the Apache parquet-testing fixtures.  Decimal / join / sort / filter semantics are
NOT pinned by any in-repo vector ("parity unpinned" for those rows; see DESIGN.md).
"""
import numpy as np

# same numeric codes as include/b200sql.h b2_dtype (GpuColumnVector.java:417-453 type map)
BOOL8, INT8, INT16, INT32, INT64, FLOAT32, FLOAT64, DATE32, TIMESTAMP_US, DECIMAL32, DECIMAL64, DECIMAL128, STRING = range(13)
_NP = {BOOL8: np.int8, INT8: np.int8, INT16: np.int16, INT32: np.int32, INT64: np.int64, FLOAT32: np.float32,
       FLOAT64: np.float64, DATE32: np.int32, TIMESTAMP_US: np.int64}
_INT_BITS = {INT8: 8, INT16: 16, INT32: 32, INT64: 64, DATE32: 32, TIMESTAMP_US: 64}


def is_decimal(dt):
    return dt in (DECIMAL32, DECIMAL64, DECIMAL128)


def decimal_dtype_for(p):  # DecimalUtil.scala:24-40
    return DECIMAL32 if p <= 9 else (DECIMAL64 if p <= 18 else DECIMAL128)


class OCol:
    """values: numpy array (object array of python ints for decimals), valid: bool array, typ=(dtype, precision, scale)"""

    def __init__(self, values, valid, typ):
        self.values = values
        self.valid = np.asarray(valid, dtype=bool)
        self.typ = tuple(typ)

    def __len__(self):
        return len(self.values)

    def to_pylist(self):
        dt = self.typ[0]
        out = []
        for v, ok in zip(self.values, self.valid):
            if not ok:
                out.append(None)
            elif dt == BOOL8:
                out.append(bool(v))
            elif dt in (FLOAT32, FLOAT64):
                out.append(float(v))
            elif dt == STRING:
                out.append(v.decode("utf-8", "replace") if isinstance(v, bytes) else v)
            else:
                out.append(int(v))
        return out


def ocol(values, typ, valid=None):
    dt = typ[0] if isinstance(typ, tuple) else typ
    typ = typ if isinstance(typ, tuple) else (typ, 0, 0)
    n = len(values)
    if valid is None:
        valid = np.array([v is not None for v in values], dtype=bool) if isinstance(values, list) else np.ones(n, bool)
    if isinstance(values, list):
        fill = b"" if dt == STRING else 0
        values = [fill if v is None else v for v in values]
    if is_decimal(dt) or dt == STRING:
        arr = np.empty(n, dtype=object)
        for i, v in enumerate(values):
            arr[i] = v if dt != STRING else (v.encode() if isinstance(v, str) else v)
            if dt != STRING:
                arr[i] = int(v)
    else:
        arr = np.asarray(values).astype(_NP[dt])
    return OCol(arr, valid, typ)


# ------------------------------------------------------------------------------------------------
# decimal type rules (Spark DecimalPrecision / DecimalType.adjustPrecisionScale; the reference
# relies on them in arithmetic.scala:513-640 DecimalMultiplyChecks)
def adjust_precision_scale(p, s):
    if p <= 38:
        return p, s
    int_digits = p - s
    min_scale = min(s, 6)
    return 38, max(38 - int_digits, min_scale)


_DEFAULT_PREC = {INT8: 3, INT16: 5, INT32: 10, INT64: 20}


def _as_decimal_type(t):
    return t if is_decimal(t[0]) else (decimal_dtype_for(_DEFAULT_PREC[t[0]]), _DEFAULT_PREC[t[0]], 0)


def _round_half_up_div(x, d):
    """BigDecimal.setScale(.., HALF_UP): round half away from zero"""
    q, r = divmod(abs(x), d)
    if r * 2 >= d:
        q += 1
    return -q if x < 0 else q


def _rescale(vals, valid, from_scale, to_prec, to_scale, check=True):
    out = np.empty(len(vals), dtype=object)
    ok = valid.copy()
    lim = 10 ** to_prec
    for i, v in enumerate(vals):
        v = int(v)
        if to_scale >= from_scale:
            r = v * 10 ** (to_scale - from_scale)
        else:
            r = _round_half_up_div(v, 10 ** (from_scale - to_scale))
        if check and abs(r) >= lim:
            ok[i] = False
            r = 0
        out[i] = r
    return out, ok


def _wrap(v, bits):
    v &= (1 << bits) - 1
    return v - (1 << bits) if v >= 1 << (bits - 1) else v


# ------------------------------------------------------------------------------------------------
def eval_expr(sx, cols):
    """evaluate an s-expression over a list of OCol -> OCol"""
    op = sx[0]
    n = len(cols[0]) if cols else 0
    if op == "col":
        c = cols[sx[1]]
        return OCol(c.values, c.valid, sx[2])
    if op == "lit" and sx[2][0] == STRING:
        v = sx[1]
        vals = np.empty(n, dtype=object)
        vals[:] = b"" if v is None else (v.encode() if isinstance(v, str) else v)
        return OCol(vals, np.full(n, v is not None), (STRING, 0, 0))
    if op == "lit":
        v, typ = sx[1], sx[2]
        dt = typ[0]
        if v is None and dt < 0:   # untyped NULL (CASE without ELSE)
            return OCol(np.zeros(n, dtype=np.int8), np.zeros(n, bool), typ)
        if v is None:
            vals = np.zeros(n, dtype=object if is_decimal(dt) else _NP[dt])
            return OCol(vals, np.zeros(n, bool), typ)
        if is_decimal(dt):
            vals = np.empty(n, dtype=object)
            vals[:] = int(v)
        else:
            vals = np.full(n, v, dtype=_NP[dt])
        return OCol(vals, np.ones(n, bool), typ)
    if op in ("add", "sub", "mul", "div", "mod", "pmod"):
        return _arith(op, eval_expr(sx[1], cols), eval_expr(sx[2], cols))
    if op in ("eq", "ne", "lt", "le", "gt", "ge", "eqns"):
        return _compare(op, eval_expr(sx[1], cols), eval_expr(sx[2], cols))
    if op in ("and", "or"):
        a, b = eval_expr(sx[1], cols), eval_expr(sx[2], cols)
        x, y = (a.values != 0) & a.valid, (b.values != 0) & b.valid
        if op == "and":  # Kleene: false dominates (predicates.scala:54-153)
            fa, fb = a.valid & ~x, b.valid & ~y
            r, v = x & y, (a.valid & b.valid) | fa | fb
        else:
            r, v = x | y, (a.valid & b.valid) | x | y
        return OCol((r & v).astype(np.int8), v, (BOOL8, 0, 0))
    if op == "not":
        a = eval_expr(sx[1], cols)
        return OCol(((a.values == 0) & a.valid).astype(np.int8), a.valid, (BOOL8, 0, 0))
    if op == "isnull":
        a = eval_expr(sx[1], cols)
        return OCol((~a.valid).astype(np.int8), np.ones(n, bool), (BOOL8, 0, 0))
    if op == "isnotnull":
        a = eval_expr(sx[1], cols)
        return OCol(a.valid.astype(np.int8), np.ones(n, bool), (BOOL8, 0, 0))
    if op in ("neg", "abs"):
        a = eval_expr(sx[1], cols)
        dt = a.typ[0]
        if dt in (FLOAT32, FLOAT64):
            return OCol(-a.values if op == "neg" else np.abs(a.values), a.valid, a.typ)
        if is_decimal(dt):
            vals = np.array([(-int(v) if (op == "neg" or v < 0) else int(v)) for v in a.values], dtype=object)
            return OCol(vals, a.valid, a.typ)
        with np.errstate(over="ignore"):
            vals = (-a.values) if op == "neg" else np.where(a.values < 0, -a.values, a.values)
        return OCol(vals.astype(a.values.dtype), a.valid, a.typ)
    if op == "coalesce":
        a, b = _unify(eval_expr(sx[1], cols), eval_expr(sx[2], cols))
        return OCol(np.where(a.valid, a.values, b.values), a.valid | b.valid, a.typ)
    if op == "if":
        p = eval_expr(sx[1], cols)
        a, b = _unify(eval_expr(sx[2], cols), eval_expr(sx[3], cols))
        t = p.valid & (p.values != 0)  # NULL predicate takes the else branch (GpuIf)
        return OCol(np.where(t, a.values, b.values), np.where(t, a.valid, b.valid), a.typ)
    if op == "cast":
        return _cast(eval_expr(sx[1], cols), sx[2])
    if op == "normnz":
        a = eval_expr(sx[1], cols)
        if a.typ[0] not in (FLOAT32, FLOAT64):
            return a
        v = a.values.copy()
        v[np.isnan(v)] = np.nan
        v[v == 0] = 0.0
        return OCol(v, a.valid, a.typ)
    if op in ("startswith", "endswith", "contains", "like"):
        # stringFunctions.scala:163 GpuStartsWith, :189 GpuEndsWith, :396 GpuContains, :972 GpuLike: NULL in, NULL out
        a, b = eval_expr(sx[1], cols), eval_expr(sx[2], cols)
        valid = a.valid & b.valid
        esc = sx[3] if op == "like" and len(sx) > 3 else "\\"
        fn = {"startswith": lambda x, y: x.startswith(y), "endswith": lambda x, y: x.endswith(y), "contains": lambda x, y: y in x,
              "like": lambda x, y: _like(x, y, esc)}[op]
        r = np.array([bool(ok and fn(x, y)) for x, y, ok in zip(a.values, b.values, valid)], dtype=bool) if n else np.zeros(0, bool)
        return OCol(r.astype(np.int8), valid, (BOOL8, 0, 0))
    if op == "substr":
        a = eval_expr(sx[1], cols)
        vals = np.empty(n, dtype=object)
        for i in range(n):
            vals[i] = substring_sql(a.values[i], sx[2], sx[3]) if a.valid[i] else b""
        return OCol(vals, a.valid, (STRING, 0, 0))
    if op == "in":   # GpuInSet / In: Kleene OR of equalities
        acc = None
        for lit_sx in sx[2]:
            e = ("eq", sx[1], lit_sx)
            acc = e if acc is None else ("or", acc, e)
        if acc is None:
            acc = ("ne", sx[1], sx[1])
        return eval_expr(acc, cols)
    if op == "case":   # GpuCaseWhen (conditionalExpressions.scala:322): first TRUE branch, else `else` (NULL when absent)
        tail = sx[2] if sx[2] is not None else ("lit", None, (-1, 0, 0))
        for c, v in reversed(sx[1]):
            tail = ("if", c, v, tail)
        return eval_expr(tail, cols)
    if op == "year":
        a = eval_expr(sx[1], cols)
        d = a.values.astype("datetime64[D]")
        return OCol((d.astype("datetime64[Y]").astype(np.int64) + 1970).astype(np.int32), a.valid, (INT32, 0, 0))
    raise NotImplementedError(op)


def substring_sql(b, pos, length):
    """UTF8String.substringSQL as GpuSubstring restates it (stringFunctions.scala:540-600): code points, 1-based pos,
    negative pos counts from the end"""
    s = b.decode("utf-8", "surrogateescape")
    nchars = len(s)
    start = pos + nchars if pos < 0 else (pos - 1 if pos > 0 else 0)
    end = max(0, min(start + length, 2**31 - 1))
    start = max(start, 0)
    if start >= end or start >= nchars:
        return b""
    return s[start:end].encode("utf-8", "surrogateescape")


def _like(x, pat, esc="\\"):
    """SQL LIKE on bytes (UTF-8): % any sequence, _ exactly one code point, esc escapes the next pattern character"""
    import re
    xs, ps = x.decode("utf-8", "surrogateescape"), pat.decode("utf-8", "surrogateescape")
    out, i = [], 0
    while i < len(ps):
        ch = ps[i]
        if ch == esc and i + 1 < len(ps):
            out.append(re.escape(ps[i + 1])); i += 2; continue
        out.append(".*" if ch == "%" else ("." if ch == "_" else re.escape(ch)))
        i += 1
    return re.fullmatch("".join(out), xs, flags=re.S) is not None


def _unify(a, b):
    if a.typ[0] < 0:   # untyped NULL takes its sibling's type
        return OCol(np.zeros(len(a), dtype=b.values.dtype), a.valid, b.typ), b
    if b.typ[0] < 0:
        return a, OCol(np.zeros(len(b), dtype=a.values.dtype), b.valid, a.typ)
    if is_decimal(a.typ[0]) and is_decimal(b.typ[0]):
        s = max(a.typ[2], b.typ[2])
        p = max(a.typ[1] - a.typ[2], b.typ[1] - b.typ[2]) + s
        t = (decimal_dtype_for(p), p, s)
        av, ao = _rescale(a.values, a.valid, a.typ[2], p, s, False)
        bv, bo = _rescale(b.values, b.valid, b.typ[2], p, s, False)
        return OCol(av, ao, t), OCol(bv, bo, t)
    assert a.typ[0] == b.typ[0], (a.typ, b.typ)
    return a, b


def _arith(op, a, b):
    n = len(a)
    if is_decimal(a.typ[0]) or is_decimal(b.typ[0]):
        ta, tb = _as_decimal_type(a.typ), _as_decimal_type(b.typ)
        p1, s1, p2, s2 = ta[1], ta[2], tb[1], tb[2]
        valid = a.valid & b.valid
        out = np.empty(n, dtype=object)
        if op in ("add", "sub"):
            s = max(s1, s2)
            p = max(p1 - s1, p2 - s2) + s + 1
            rp, rs = adjust_precision_scale(p, s)
            assert rs == s, "decimal add with precision loss not restated"
            lim = 10 ** rp
            for i in range(n):
                x = int(a.values[i]) * 10 ** (s - s1)
                y = int(b.values[i]) * 10 ** (s - s2)
                r = x + y if op == "add" else x - y
                if abs(r) >= lim:  # arithmetic.scala:78-125: NULL on overflow (non-ANSI)
                    valid[i] = False
                    r = 0
                out[i] = r if valid[i] else 0
            return OCol(out, valid, (decimal_dtype_for(rp), rp, rs))
        if op == "mul":  # arithmetic.scala:411-512
            p, s = p1 + p2 + 1, s1 + s2
            rp, rs = adjust_precision_scale(p, s)
            lim = 10 ** rp
            for i in range(n):
                r = int(a.values[i]) * int(b.values[i])
                if rs < s:
                    r = _round_half_up_div(r, 10 ** (s - rs))
                if abs(r) >= lim:
                    valid[i] = False
                out[i] = r if valid[i] else 0
            return OCol(out, valid, (decimal_dtype_for(rp), rp, rs))
        if op == "div":  # arithmetic.scala:903-1000 (Spark Divide result type, HALF_UP, x / 0 -> NULL)
            rs = max(6, s1 + p2 + 1)
            rp, rs = adjust_precision_scale(p1 - s1 + s2 + rs, rs)
            k = rs - s1 + s2
            lim = 10 ** rp
            for i in range(n):
                d = int(b.values[i])
                if d == 0 or not valid[i]:
                    valid[i] = False
                    out[i] = 0
                    continue
                num = int(a.values[i]) * 10 ** k
                q, r = divmod(abs(num), abs(d))
                if r * 2 >= abs(d):
                    q += 1
                q = -q if (num < 0) != (d < 0) else q
                if abs(q) >= lim or abs(q) >= 10 ** 38:
                    valid[i] = False
                    q = 0
                out[i] = q
            return OCol(out, valid, (decimal_dtype_for(rp), rp, rs))
        raise NotImplementedError("decimal " + op)
    assert a.typ[0] == b.typ[0], (a.typ, b.typ)
    dt = a.typ[0]
    valid = a.valid & b.valid
    x, y = a.values, b.values
    if dt in (FLOAT32, FLOAT64):
        with np.errstate(all="ignore"):
            if op == "add":
                r = x + y
            elif op == "sub":
                r = x - y
            elif op == "mul":
                r = x * y
            else:
                zero = y == 0
                valid = valid & ~zero  # Spark: x / 0 and x % 0 are NULL
                ys = np.where(zero, 1, y)
                if op == "div":
                    r = x / ys
                else:
                    r = np.fmod(x, ys)
                    if op == "pmod":   # Spark Pmod: r = a % n; if (r < 0) (r + n) % n else r  (arithmetic.scala:1177 BinaryOp.PMOD)
                        r = np.where(r < 0, np.fmod(r + ys, ys), r)
                r = np.where(zero, 0, r)
        return OCol(r.astype(x.dtype), valid, a.typ)
    bits = _INT_BITS[dt]
    with np.errstate(over="ignore"):
        if op == "add":
            r = x + y
        elif op == "sub":
            r = x - y
        elif op == "mul":
            r = x * y
        else:
            zero = y == 0
            valid = valid & ~zero
            ys = np.where(zero, 1, y).astype(object)
            xs = x.astype(object)
            res = np.empty(n, dtype=object)
            for i in range(n):
                xi, yi = int(xs[i]), int(ys[i])
                q = abs(xi) // abs(yi)
                q = q if (xi < 0) == (yi < 0) else -q  # Java: truncate toward zero
                if op == "div":
                    res[i] = _wrap(q, bits)
                else:
                    rem = xi - q * yi
                    if op == "pmod" and rem < 0:   # (r + n) % n, the add wrapping in the operand type (int/long; byte/short add as int)
                        s2 = _wrap(rem + yi, max(bits, 32))
                        q2 = abs(s2) // abs(yi)
                        q2 = q2 if (s2 < 0) == (yi < 0) else -q2
                        rem = s2 - q2 * yi
                    res[i] = _wrap(rem, bits)
            r = np.where(zero, 0, res).astype(x.dtype)
    return OCol(r.astype(x.dtype), valid, a.typ)


def _cmp3(x, y, is_float):
    """-1/0/1 with Spark float order: NaN == NaN, NaN greatest, -0.0 == 0.0 (predicates.scala:155-331)"""
    if is_float:
        xn, yn = np.isnan(x), np.isnan(y)
        with np.errstate(invalid="ignore"):
            c = np.where(x < y, -1, np.where(x > y, 1, 0))
        c = np.where(xn & yn, 0, np.where(xn, 1, np.where(yn, -1, c)))
        return c
    return np.where(x < y, -1, np.where(x > y, 1, 0))


def _compare(op, a, b):
    a, b = _unify(a, b)
    dt = a.typ[0]
    if dt == STRING:
        c = np.array([(-1 if x < y else (1 if x > y else 0)) for x, y in zip(a.values, b.values)])
    else:
        c = _cmp3(a.values, b.values, dt in (FLOAT32, FLOAT64))
    c = c.astype(np.int64)
    valid = a.valid & b.valid
    if op == "eqns":
        r = np.where(valid, c == 0, a.valid == b.valid)
        return OCol(r.astype(np.int8), np.ones(len(a), bool), (BOOL8, 0, 0))
    r = {"eq": c == 0, "ne": c != 0, "lt": c < 0, "le": c <= 0, "gt": c > 0, "ge": c >= 0}[op]
    return OCol((r & valid).astype(np.int8), valid, (BOOL8, 0, 0))


def _cast(a, to):
    to = tuple(to)
    fdt, tdt = a.typ[0], to[0]
    n = len(a)
    if fdt == tdt and (not is_decimal(tdt) or a.typ[1:] == to[1:]):
        return a
    if is_decimal(tdt):
        ft = _as_decimal_type(a.typ)
        vals, ok = _rescale(a.values, a.valid, ft[2], to[1], to[2], True)
        return OCol(vals, ok, (tdt, to[1], to[2]))
    if is_decimal(fdt):
        assert tdt in (FLOAT32, FLOAT64)
        v = np.array([int(x) for x in a.values], dtype=np.float64) / (10.0 ** a.typ[2])
        return OCol(v.astype(_NP[tdt]), a.valid, (tdt, 0, 0))
    x = a.values
    if tdt == BOOL8:
        return OCol((x != 0).astype(np.int8), a.valid, (BOOL8, 0, 0))
    if fdt in (FLOAT32, FLOAT64) and tdt not in (FLOAT32, FLOAT64):
        # Java (int)/(long) conversion: NaN -> 0, saturating; byte/short narrow from int
        wide_bits = 64 if _INT_BITS[tdt] == 64 else 32
        lo, hi = -(1 << (wide_bits - 1)), (1 << (wide_bits - 1)) - 1
        out = np.empty(n, dtype=object)
        for i in range(n):
            f = float(x[i])
            if f != f:
                v = 0
            elif f >= hi:
                v = hi
            elif f <= lo:
                v = lo
            else:
                v = int(f)
            out[i] = _wrap(v, _INT_BITS[tdt])
        return OCol(out.astype(_NP[tdt]), a.valid, (tdt, 0, 0))
    with np.errstate(all="ignore"):
        return OCol(x.astype(_NP[tdt]), a.valid, (tdt, 0, 0))


# ------------------------------------------------------------------------------------------------
# filter (basicPhysicalOperators.scala:1148-1224): NULL predicate drops the row; order preserved
def filter_cols(cols, pred):
    keep = pred.valid & (pred.values != 0)
    return [OCol(c.values[keep], c.valid[keep], c.typ) for c in cols]


# ------------------------------------------------------------------------------------------------
# aggregates.  spec = (kind, column, out_dtype, out_scale, out_precision); kinds as b2_agg_kind
AGG_SUM, AGG_COUNT, AGG_MIN, AGG_MAX, AGG_COUNT_ALL = 1, 2, 3, 4, 5


def _agg_one(kind, col, rows, spec):
    """aggregate the given row indexes of col -> (value, valid)"""
    if kind == AGG_COUNT_ALL:
        return len(rows), True
    vals, ok = col.values[rows], col.valid[rows]
    if kind == AGG_COUNT:  # aggregateFunctions.scala:1408-1432: non-null count, never null
        return int(ok.sum()), True
    sel = vals[ok]
    if len(sel) == 0:
        return 0, False  # empty / all-null group -> NULL (isEmpty protocol, :1106-1190)
    dt = col.typ[0]
    if kind == AGG_SUM:
        if dt in (FLOAT32, FLOAT64):
            import math
            return math.fsum(float(v) for v in sel), True  # exactly rounded sum = the <=1ulp target
        s = sum(int(v) for v in sel)
        if is_decimal(dt):
            if abs(s) >= 10 ** spec[4]:  # GpuCheckOverflowAfterSum (:820): NULL when out of precision
                return 0, False
            return s, True
        return _wrap(s, 64), True  # long sum wraps (:1041-1104, non-ANSI)
    if dt in (FLOAT32, FLOAT64):  # NaN is the largest value (:368-465, 546-600)
        nan = np.isnan(sel.astype(np.float64))
        if kind == AGG_MAX:
            return (float("nan"), True) if nan.any() else (float(sel.max()), True)
        rest = sel[~nan]
        return (float("nan"), True) if len(rest) == 0 else (float(rest.min()), True)
    return (min(sel) if kind == AGG_MIN else max(sel)), True


def _out_type(spec, col):
    kind = spec[0]
    if kind in (AGG_COUNT, AGG_COUNT_ALL):
        return (INT64, 0, 0)
    if kind in (AGG_MIN, AGG_MAX):
        return col.typ
    if kind == AGG_SUM and col.typ[0] in (FLOAT32, FLOAT64):
        return (spec[2], 0, 0)
    return (spec[2], spec[4] if len(spec) > 4 else 0, spec[3])


def reduce_cols(cols, specs):
    """AggHelper.performReduction: one output row; empty input -> sum NULL, count 0 (GpuAggregateExec.scala:1107-1126)"""
    n = len(cols[0]) if cols else 0
    rows = np.arange(n)
    out = []
    for spec in specs:
        col = cols[spec[1]] if spec[0] != AGG_COUNT_ALL else None
        v, ok = _agg_one(spec[0], col, rows, spec)
        out.append(ocol([v], _out_type(spec, col), np.array([ok])))
    return out


def _key_of(col, i):
    if not col.valid[i]:
        return None  # NULL is its own group (GpuAggregateExec.scala:565-568)
    v = col.values[i]
    if col.typ[0] in (FLOAT32, FLOAT64):
        f = float(v)
        if f != f:
            return "nan"  # NaN == NaN
        return 0.0 if f == 0 else f  # -0.0 == 0.0
    return v if col.typ[0] == STRING else int(v)


def _normalized_key_values(col, rows):
    """the key values of the given representative rows; floating-point keys come out as +0.0 for -0.0 and the canonical NaN
    for every NaN, as Spark normalises grouping keys before aggregating (NormalizeFloatingNumbers.scala:29-38)"""
    vals = col.values[rows]
    if col.typ[0] in (FLOAT32, FLOAT64):
        with np.errstate(invalid="ignore"):   # signalling NaN payloads
            vals = np.where(np.isnan(vals), np.array(np.nan, vals.dtype), vals + np.array(0.0, vals.dtype)).astype(vals.dtype)
    return vals


def groupby_cols(cols, key_idx, specs):
    """AggHelper.performGroupByAggregation: keys then aggregates; group order = first appearance
    (callers compare order-insensitively: output order is unspecified in the reference)"""
    n = len(cols[0]) if cols else 0
    groups = {}
    for i in range(n):
        k = tuple(_key_of(cols[c], i) for c in key_idx)
        groups.setdefault(k, []).append(i)
    firsts = [rows[0] for rows in groups.values()]
    out = [OCol(_normalized_key_values(cols[c], firsts), cols[c].valid[firsts], cols[c].typ) for c in key_idx]
    for spec in specs:
        col = cols[spec[1]] if spec[0] != AGG_COUNT_ALL else None
        vals, oks = [], []
        for rows in groups.values():
            v, ok = _agg_one(spec[0], col, np.array(rows), spec)
            vals.append(v)
            oks.append(ok)
        out.append(ocol(vals, _out_type(spec, col), np.array(oks, dtype=bool)))
    return out


def rows_of(cols):
    lists = [c.to_pylist() for c in cols]
    return list(zip(*lists)) if lists else []


def sort_rows_for_compare(rows):
    """order-insensitive comparison key (the reference sorts locally before comparing:
    SparkQueryCompareTestSuite.scala:884-918)"""
    def k(r):
        return tuple((0, "") if v is None else ((2, "nan") if isinstance(v, float) and v != v else (1, v)) for v in r)
    return sorted(rows, key=lambda r: tuple(str(type(x[1])) + repr(x) for x in k(r)))
