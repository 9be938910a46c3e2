"""Generated row code at every numeric type's boundary values, against an exact reference kept in this file.

The reference restates DESIGN.md §4.5 in plain Python: the coercion lattice, casts that fail to NULL, integer
arithmetic that wraps in the coerced type, a truncating divide whose zero divisor in a valid slot is an error, single
IEEE float operations, and sum / min / max / count.  Python integers and numpy scalars make it exact, so results are
compared bit for bit (NaN by NaN-ness only; its payload after arithmetic is not specified).  Float sums are checked
against math.fsum with the order-free bound |got - exact| <= (n - 1) u_T sum|x|.  The CPU oracle is a second anchor: the
reference must agree with it on every projection and aggregate checked here.

Data: 13 boundary values per type, laid out as a strength-2 orthogonal array over GF(13) (block row (a, b), column c
holds value index a + c b mod 13).  Any two columns meet every pair of values exactly once in the 169-row block.  The
block is repeated to an odd length, so full staged tiles, the vector tail and the row tail all see every combination,
while the reference runs on the 169 block rows.
"""
import math

import numpy as np
import pytest

from fuse_query_b200 import cabi
from oracle import binding as o

pytestmark = pytest.mark.gpu

TYPES = ["i8", "i16", "i32", "i64", "u8", "u16", "u32", "u64", "f32", "f64"]
TAG = {"i8": cabi.I8, "i16": cabi.I16, "i32": cabi.I32, "i64": cabi.I64, "u8": cabi.U8, "u16": cabi.U16, "u32": cabi.U32,
       "u64": cabi.U64, "f32": cabi.F32, "f64": cabi.F64, "bool": cabi.BOOL}
NP = {"i8": np.int8, "i16": np.int16, "i32": np.int32, "i64": np.int64, "u8": np.uint8, "u16": np.uint16, "u32": np.uint32,
      "u64": np.uint64, "f32": np.float32, "f64": np.float64, "bool": np.uint8}
UINT = {"f32": np.uint32, "f64": np.uint64}
BITS = {"i8": 8, "i16": 16, "i32": 32, "i64": 64, "u8": 8, "u16": 16, "u32": 32, "u64": 64}
ORDER = ["f64", "f32", "i64", "i32", "i16", "i8", "u64", "u32", "u16", "u8"]   # codegen.cc numerical_coercion
UNIT_ROUNDOFF = {"f32": 2.0 ** -24, "f64": 2.0 ** -53}
DIVZERO = "Internal Error: Divide by zero error"
ARITH = ["+", "-", "*", "/"]
CMPS = ["=", "<", "<=", ">", ">="]

INF, NAN = math.inf, math.nan
F32_MAX, F64_MAX = float(np.finfo(np.float32).max), float(np.finfo(np.float64).max)
BOUNDARY = {
    "i8": [0, 1, -1, -128, -127, 126, 127, 2, -2, 63, -64, 100, -100],
    "i16": [0, 1, -1, -32768, -32767, 32766, 32767, 127, 128, 255, 256, -128, -129],
    "i32": [0, 1, -1, -2**31, -2**31 + 1, 2**31 - 2, 2**31 - 1, 32767, 32768, 65535, 65536, -32768, -32769],
    "i64": [0, 1, -1, -2**63, -2**63 + 1, 2**63 - 2, 2**63 - 1, 2**31 - 1, 2**31, 2**32 - 1, 2**32,
            2**60 + 2**36 + 1, 2**53 + 1],                                   # the last two round when cast to f32 / f64
    # unsigned values sit on both sides of every signed MAX they can be cast to (a cast fails at exactly MAX + 1)
    "u8": [0, 1, 254, 255, 127, 128, 2, 3, 100, 200, 64, 129, 126],
    "u16": [0, 1, 65534, 65535, 127, 128, 32767, 32768, 255, 256, 200, 1000, 2049],
    "u32": [0, 1, 2**32 - 2, 2**32 - 1, 127, 128, 32767, 32768, 2**31 - 1, 2**31, 2**24 + 1, 65535, 255],
    "u64": [0, 1, 2**64 - 2, 2**64 - 1, 127, 128, 32767, 32768, 2**31 - 1, 2**31, 2**63 - 1, 2**63,
            2**64 - 2**39 - 1],                                              # to f32 in one rounding: 2^64 - 2^40, not 2^64
    "f32": [0.0, -0.0, 1.0, -1.0, INF, -INF, F32_MAX, -F32_MAX, 2.0**-149, -2.0**-149, NAN, 1.5, 2.0**-126],
    "f64": [0.0, -0.0, 1.0, -1.0, INF, -INF, F64_MAX, -F64_MAX, 5e-324, -5e-324, NAN, 2.0**53 + 2, 0.1],
}
# float values for sums and min/max: finite, no NaN, far enough below MAX that 10^5 of them cannot overflow
AGG_FLOATS = [0.0, -0.0, 1.0, -1.0, 0.5, -2.0, 1.5, 3.0, -0.1, 1e6, -1e6, 2.0**-20, 7.25]

Q = 13
BLOCK = Q * Q
REPS = 593                       # odd: 100 217 rows
N = BLOCK * REPS
OA_A = np.repeat(np.arange(Q), Q)
OA_B = np.tile(np.arange(Q), Q)


def oa_index(c):
    """value index of OA column c in each block row"""
    return (OA_A + c * OA_B) % Q


# ---------------------------------------------------------------------------------------------
# the reference (DESIGN.md §4.5)
# ---------------------------------------------------------------------------------------------
class DivZero(Exception):
    pass


def is_float(t):
    return t[0] == "f"


def int_range(t):
    b = BITS[t]
    return (-(1 << (b - 1)), (1 << (b - 1)) - 1) if t[0] == "i" else (0, (1 << b) - 1)


def coerce(l, r):
    return l if l == r else next(t for t in ORDER if t in (l, r))


def wrap(v, t):
    b = BITS[t]
    v &= (1 << b) - 1
    return v - (1 << b) if t[0] == "i" and v >= 1 << (b - 1) else v


def int_to_float(v, t):
    """an integer rounded once to the nearest float of type t (ties to even)"""
    if t == "f64":
        return np.float64(float(v))          # Python's int -> float conversion is correctly rounded
    m, e = abs(v), abs(v).bit_length() - 24
    if e > 0:
        q, r = divmod(m, 1 << e)
        if r > 1 << (e - 1) or (r == 1 << (e - 1) and q & 1):
            q += 1
        m = q << e
    return np.float32(-m if v < 0 else m)    # exact: m has at most 24 significant bits


def cast(x, s, t):
    """-> (value, representable).  Coercion never narrows a float, so s is an integer or f32 -> f64."""
    if s == t:
        return x, True
    if is_float(t):
        return (np.float64(x), True) if is_float(s) else (int_to_float(x, t), True)
    lo, hi = int_range(t)
    return (x, True) if lo <= x <= hi else (0, False)


def arith(op, a, b, t):
    if is_float(t):
        with np.errstate(all="ignore"):
            return {"+": np.add, "-": np.subtract, "*": np.multiply, "/": np.divide}[op](a, b)
    if op == "/":
        q = abs(a) // abs(b)
        return wrap(q if (a < 0) == (b < 0) else -q, t)     # truncates toward zero; MIN / -1 wraps to MIN
    return wrap({"+": a + b, "-": a - b, "*": a * b}[op], t)


def compare(op, a, b):
    return bool({"=": a == b, "<": a < b, "<=": a <= b, ">": a > b, ">=": a >= b}[op])


def parse(sexpr):
    toks = sexpr.replace("(", " ( ").replace(")", " ) ").split()

    def rd(i):
        assert toks[i] == "("
        out, i = [], i + 1
        while toks[i] != ")":
            if toks[i] == "(":
                x, i = rd(i)
                out.append(x)
            else:
                out.append(toks[i])
                i += 1
        return out, i + 1
    return rd(0)[0]


def literal(t, text):
    if is_float(t):
        return NP[t](float(text))
    return int(text)


def evaluate(node, row, table):
    """-> (value, valid, type) of an expression at one block row"""
    head = node[0]
    if head == "col":
        c = table[node[1]]
        return c.block[row], c.block_ok[row], c.t
    if head in NP:
        return literal(head, node[1]), True, head
    lv, lok, lt = evaluate(node[1], row, table)
    rv, rok, rt = evaluate(node[2], row, table)
    if head in ("and", "or"):
        return (lv and rv) if head == "and" else (lv or rv), lok and rok, "bool"
    t = coerce(lt, rt)
    a, ka = cast(lv, lt, t)
    b, kb = cast(rv, rt, t)
    ok = lok and rok and ka and kb
    if head in CMPS:
        return compare(head, a, b), ok, "bool"
    if head == "/" and b == 0:
        if ok:
            raise DivZero()
        return NP[t](0) if is_float(t) else 0, False, t
    return arith(head, a, b, t), ok, t


def reference(expr, table):
    """-> (values, valid, type) over the block rows"""
    node = parse(expr)
    vals, oks = [], []
    for r in range(BLOCK):
        v, ok, t = evaluate(node, r, table)
        vals.append(v if ok else (NP[t](0) if is_float(t) else 0))
        oks.append(ok)
    return vals, np.array(oks), t


def as_numpy(vals, t):
    if t == "bool":
        return np.array([1 if v else 0 for v in vals], dtype=np.uint8)
    if is_float(t):
        return np.array(vals, dtype=NP[t])
    return np.array([int(v) for v in vals], dtype=object).astype(NP[t])


def same_values(got, want, t):
    """bits for integers and floats, NaN-ness only for NaN"""
    if not is_float(t):
        return np.array_equal(got.astype(NP[t]), want.astype(NP[t]))
    gn, wn = np.isnan(got), np.isnan(want)
    return np.array_equal(gn, wn) and np.array_equal(got[~gn].view(UINT[t]), want[~wn].view(UINT[t]))


# ---------------------------------------------------------------------------------------------
# the table
# ---------------------------------------------------------------------------------------------
class Col:
    def __init__(self, name, t, block=None, block_ok=None, full=None, valid_kind=None):
        self.name, self.t = name, t
        self.block = block                                  # block values (Python ints / numpy floats), or None
        self.block_ok = block_ok if block_ok is not None else [True] * BLOCK
        self.full = full                                    # N values of a column that does not repeat the block
        self.valid_kind = valid_kind                        # None, "bytes" or "bitmap"

    def values(self):
        return self.full if self.full is not None else np.tile(as_numpy(self.block, self.t), REPS)

    def nullable(self):
        return 1 if self.valid_kind == "bytes" else 2 if self.valid_kind == "bitmap" else 0


BITMAP_OFFSET = 5
NULL_ROWS = (np.arange(BLOCK) * 7) % 5 == 0               # NULL slots of the nullable copies: 34 of 169 block rows


def make_table():
    tbl = {}
    for k, t in enumerate(TYPES):
        vals = BOUNDARY[t] if not is_float(t) else [NP[t](v) for v in BOUNDARY[t]]
        for name, c in ((f"x_{t}", k), (f"y_{t}", (k + 10) % Q)):
            block = [vals[i] for i in oa_index(c)]
            tbl[name] = Col(name, t, block)
            # divisor copy: zero slots (0, 0.0, -0.0) are NULL
            tbl["d" + name] = Col("d" + name, t, block, [v != 0 for v in block], valid_kind="bytes")
        # nullable copy; Int16's validity is an Arrow bitmap that starts at a bit offset
        tbl[f"n_{t}"] = Col(f"n_{t}", t, tbl[f"x_{t}"].block, list(~NULL_ROWS), valid_kind="bitmap" if t == "i16" else "bytes")
    for k, t in ((8, "f32"), (9, "f64")):
        agg = [NP[t](v) for v in AGG_FLOATS]
        tbl[f"a_{t}"] = Col(f"a_{t}", t, [agg[i] for i in oa_index(k)], list(~NULL_ROWS), valid_kind="bytes")
        # min / max inputs: the boundary values without NaN
        tbl[f"m_{t}"] = Col(f"m_{t}", t, [v if not np.isnan(v) else NP[t](2.0) for v in tbl[f"x_{t}"].block])
    rng = np.random.default_rng(2026)
    tbl["s"] = Col("s", "u32", full=rng.integers(0, 1 << 32, N, dtype=np.uint64).astype(np.uint32))
    tbl["z"] = Col("z", "u8", full=np.zeros(N, np.uint8))
    for t in ("f32", "f64"):
        tbl[f"r_{t}"] = Col(f"r_{t}", t, full=rng.normal(0, 1000, N).astype(NP[t]))
        for j in range(3):
            tbl[f"fma{j}_{t}"] = Col(f"fma{j}_{t}", t, full=rng.normal(0, 1, N).astype(NP[t]))
    return tbl


TABLE = make_table()


def tiled_valid(c):
    return np.tile(np.array(c.block_ok, dtype=np.uint8), REPS) if c.full is None else np.ones(N, np.uint8)


@pytest.fixture(scope="module")
def env():
    ctx = cabi.Context(0)
    dev = {}
    for name, c in TABLE.items():
        v = c.values()
        if c.valid_kind == "bytes":
            dev[name] = ctx.from_numpy(v, tiled_valid(c))
        elif c.valid_kind == "bitmap":
            bits = np.concatenate([np.zeros(BITMAP_OFFSET, np.uint8), tiled_valid(c)])
            dev[name] = ctx.from_numpy(v, valid_bitmap=np.packbits(bits, bitorder="little"), bit_offset=BITMAP_OFFSET)
        else:
            dev[name] = ctx.from_numpy(v)
    yield ctx, dev
    ctx.close()


def columns_of(exprs):
    cols = []
    for e in exprs:
        toks = e.replace("(", " ").replace(")", " ").split()
        for i, tok in enumerate(toks[:-1]):
            if tok == "col" and toks[i + 1] not in cols:
                cols.append(toks[i + 1])
    return cols


def packs(exprs, fixed_cols=()):
    """expressions in pipes of at most 8 select expressions over at most 8 columns"""
    out, cur = [], []
    for e in exprs:
        cand = cur + [e]
        if len(cand) > 8 or len(set(columns_of(cand)) | set(fixed_cols)) > 8:
            out.append(cur)
            cand = [e]
        cur = cand
    return out + ([cur] if cur else [])


def pipe_for(ctx, exprs, cols, **kw):
    return ctx.pipe(exprs, columns=cols, dtypes=[TAG[TABLE[c].t] for c in cols], nullable=[TABLE[c].nullable() for c in cols], **kw)


def run_project(env, exprs, predicate=None):
    ctx, dev = env
    cols = columns_of(([predicate] if predicate else []) + exprs)
    pipe = pipe_for(ctx, exprs, cols, predicate=predicate)
    outs = [ctx.column(pipe.expr_dtype(i), N) for i in range(len(exprs))]
    ov = [ctx.column(cabi.BOOL, N) if pipe.expr_nullable(i) else None for i in range(len(exprs))]
    pipe.launch_project(cabi.make_source([dev[c] for c in cols], N), outs, N, out_valid=ov)
    sel, written = pipe.fetch_project()
    assert sel == written
    res = [(pipe.expr_dtype(i), outs[i].to_numpy(written), None if ov[i] is None else ov[i].to_numpy(written)) for i in range(len(exprs))]
    for c in outs + [v for v in ov if v is not None]:
        c.free()
    pipe.destroy()
    return res, written


def check_projection(env, exprs, predicate=None, rows=None):
    """run `exprs` (packed into pipes) and compare every output row with the reference; rows = kept source rows"""
    rows = np.arange(N) if rows is None else rows
    for pack in packs(exprs, columns_of([predicate]) if predicate else ()):
        got, written = run_project(env, pack, predicate)
        assert written == len(rows), (pack, predicate, written, len(rows))
        for e, (dtype, vals, valid) in zip(pack, got):
            wv, wok, t = reference(e, TABLE)
            assert dtype == TAG[t], (e, dtype, t)
            want_ok = wok[rows % BLOCK]
            if valid is None:
                assert want_ok.all(), f"{e}: NULL slots but no validity output"
                keep = np.ones(len(rows), bool)
            else:
                assert np.array_equal(valid.astype(bool), want_ok), f"validity of {e}"
                keep = want_ok
            want = as_numpy(wv, t)[rows % BLOCK]
            assert same_values(vals[keep], want[keep], t), (e, vals[keep][:20], want[keep][:20])


# ---------------------------------------------------------------------------------------------
# the expressions
# ---------------------------------------------------------------------------------------------
def pair_columns(l, r):
    """left, right and divisor columns of the pair (l, r): distinct OA columns, so every value pair meets"""
    if l == r:
        return f"x_{l}", f"y_{r}", f"dy_{r}"
    return f"x_{l}", f"x_{r}", f"dx_{r}"


def binary_ops(left, right, divisor):
    return [f"({op} (col {left}) (col {divisor if op == '/' else right}))" for op in ARITH] + \
           [f"({op} (col {left}) (col {right}))" for op in CMPS]


def matrix_exprs(l):
    out = []
    for r in TYPES:
        out += binary_ops(*pair_columns(l, r))
    return out


def literal_text(t, v):
    return repr(float(v)) if is_float(t) else str(int(v))


def literal_exprs(t):
    """each boundary literal of type t on both sides of an arithmetic operator with a column of type t, and in one
    comparison with a column of another type"""
    out = []
    k = TYPES.index(t)
    for i, v in enumerate(BOUNDARY[t]):
        lit = f"({t} {literal_text(t, v)})"
        op_r = ARITH[i % 4] if not (ARITH[i % 4] == "/" and v == 0) else "+"    # a constant zero divisor is its own case
        op_l = ARITH[(i + 1) % 4]
        out.append(f"({op_r} (col x_{t}) {lit})")
        out.append(f"({op_l} {lit} (col {'dx_' + t if op_l == '/' else 'y_' + t}))")
        other = TYPES[(k + 1 + i) % len(TYPES)]
        out.append(f"({CMPS[i % 5]} {lit} (col x_{other}))")
    return out


PARTNER = {"i8": "u64", "i16": "u8", "i32": "u16", "i64": "u32", "u8": "u8", "u16": "u8", "u32": "u16", "u64": "u32",
           "f32": "i64", "f64": "u64"}


def sink_pair(t, agg=False):
    """one operand pair whose coerced type is t; the left operand is a nullable column"""
    p = PARTNER[t]
    assert coerce(t, p) == t
    left = f"a_{t}" if agg and is_float(t) else f"n_{t}"
    right, div = (f"y_{t}", f"dy_{t}") if p == t else (f"x_{p}", f"dx_{p}")
    return left, right, div


# ---------------------------------------------------------------------------------------------
# the reference against the CPU oracle (second anchor)
# ---------------------------------------------------------------------------------------------
def oracle_table(cols):
    out = {}
    for c in cols:
        col = TABLE[c]
        valid = None if col.valid_kind is None else np.array(col.block_ok, np.uint8)
        out[c] = o.Array(TAG[col.t], as_numpy(col.block, col.t), valid)
    return out


def test_reference_agrees_with_the_oracle():
    exprs = [e for t in TYPES for e in matrix_exprs(t) + literal_exprs(t)]
    exprs += [e for t in TYPES for e in binary_ops(*sink_pair(t))]
    for e in exprs:
        vals, ok, t = reference(e, TABLE)
        try:
            c = o.run_query([e], table=oracle_table(columns_of([e])), worker_threads=1, tail_quirk=False).columns[0]
        except o.OracleError as err:
            # The one known deviation: the reference converts a comparison's literal to the lane type with `try_into()?`
            # (macros.rs:85-96), so a literal that does not fit raises.  The device applies the cast rule of
            # DESIGN.md §4.5 to the literal like to any operand: every slot is NULL.
            assert str(err).startswith("Internal Error: Cannot convert NULL to ") and parse(e)[0] in CMPS and not ok.any(), (e, str(err))
            continue
        assert c.dtype == TAG[t], (e, c.dtype, t)
        ook = np.ones(BLOCK, bool) if c.valid is None else c.valid.astype(bool)
        assert np.array_equal(ook, ok), f"validity of {e}"
        assert same_values(c.values[ok], as_numpy(vals, t)[ok], t), e


def test_single_rounding_of_integers_to_float():
    assert int_to_float(2**60 + 2**36 + 1, "f32") == 2.0**60 + 2.0**37
    assert np.float32(float(2**60 + 2**36 + 1)) == 2.0**60       # what rounding twice through f64 would give
    assert int_to_float(2**64 - 2**39 - 1, "f32") == 2.0**64 - 2.0**40
    assert int_to_float(2**53 + 1, "f64") == 2.0**53
    vals = np.array([v for v in BOUNDARY["i64"]], dtype=np.int64)
    assert np.array_equal(vals.astype(np.float32), np.array([int_to_float(v, "f32") for v in BOUNDARY["i64"]], np.float32))


# ---------------------------------------------------------------------------------------------
# projection without a filter (map kernel): every ordered pair of types, every literal, contraction
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("left", TYPES)
def test_projection_every_type_pair(env, left):
    check_projection(env, matrix_exprs(left))


@pytest.mark.parametrize("t", TYPES)
def test_projection_boundary_literals(env, t):
    check_projection(env, literal_exprs(t))


def test_projection_is_not_contracted_into_fma(env):
    """a * b + c and a * b - c round twice (random normals: almost every product is inexact)"""
    exprs, want = [], []
    for t in ("f32", "f64"):
        a, b, c = (TABLE[f"fma{j}_{t}"].full for j in range(3))
        exprs += [f"(+ (* (col fma0_{t}) (col fma1_{t})) (col fma2_{t}))", f"(- (* (col fma0_{t}) (col fma1_{t})) (col fma2_{t}))"]
        want += [(a * b) + c, (a * b) - c]
    got, written = run_project(env, exprs)
    assert written == N
    for e, (_, vals, _), w in zip(exprs, got, want):
        assert vals.dtype == w.dtype and same_values(vals, w, "f32" if w.dtype == np.float32 else "f64"), e


# ---------------------------------------------------------------------------------------------
# filter + projection
# ---------------------------------------------------------------------------------------------
HALF = "(< (col s) (u32 2147483648))"
FEW = "(and (< (col s) (u32 33554432)) (<= (col n_i16) (col x_u8)))"     # NULL through the bitmap column: the row is dropped


def kept_rows(predicate):
    s = TABLE["s"].full
    if predicate == HALF:
        return np.nonzero(s < 2147483648)[0]
    vals, ok, _ = reference("(<= (col n_i16) (col x_u8))", TABLE)
    cmp_ = np.array(vals, bool) & ok
    return np.nonzero((s < 33554432) & cmp_[np.arange(N) % BLOCK])[0]


@pytest.mark.parametrize("predicate", [HALF, FEW], ids=["half", "few"])
def test_filter_and_projection(env, predicate):
    rows = kept_rows(predicate)
    assert (0.4 * N < len(rows) < 0.6 * N) if predicate == HALF else (50 < len(rows) < 0.01 * N)
    exprs = [e for t in TYPES for e in binary_ops(*sink_pair(t))]
    check_projection(env, exprs, predicate, rows)


# ---------------------------------------------------------------------------------------------
# aggregates
# ---------------------------------------------------------------------------------------------
def agg_reference(op, vals, ok, t, reps=REPS):
    """sum / min / max / count of a repeated block -> (value | None, n valid, sum |x|)"""
    if op == "count":
        return len(vals) * reps, None, None
    v = [x for x, k in zip(vals, ok) if k]
    if not v:
        return None, 0, None
    if op == "min":
        return min(v), len(v), None
    if op == "max":
        return max(v), len(v), None
    if is_float(t):
        return math.fsum([float(x) for x in v] * reps), len(v) * reps, math.fsum(abs(float(x)) for x in v) * reps
    return wrap(sum(int(x) for x in v) * reps, t), len(v) * reps, None


def check_agg_value(e, got, want, n, abs_sum, t, op):
    if want is None:
        assert got is None, (e, got)
        return
    if op == "sum" and is_float(t):
        assert abs(got - want) <= (n - 1) * UNIT_ROUNDOFF[t] * abs_sum, (e, got, want)
    elif is_float(t):
        assert got == float(want), (e, got, want)      # ±0.0 tie: which zero min/max keeps depends on the fold order
    else:
        assert got == want, (e, got, want)


def run_aggregate(env, exprs):
    ctx, dev = env
    cols = columns_of(exprs)
    pipe = pipe_for(ctx, exprs, cols, aggregate=True)
    pipe.launch_aggregate(cabi.make_source([dev[c] for c in cols], N))
    states, rows = pipe.fetch_aggregate()
    pipe.destroy()
    assert rows == N
    return states


def parse_arg(e):
    return e[e.index(" ") + 1:-1]


def agg_exprs_over_pairs(t):
    left, right, div = sink_pair(t, agg=True)
    out = []
    for op in ARITH:
        arg = f"({op} (col {left}) (col {div if op == '/' else right}))"
        out += [f"({a} {arg})" for a in ("sum", "min", "max", "count")]
    return out


def agg_exprs_over_columns(t):
    if is_float(t):
        return [f"(sum (col a_{t}))", f"(sum (col r_{t}))", f"(min (col m_{t}))", f"(max (col m_{t}))", f"(count (col x_{t}))",
                f"(max (col a_{t}))"]
    return [f"(sum (col x_{t}))", f"(sum (col n_{t}))", f"(min (col n_{t}))", f"(max (col x_{t}))", f"(count (col n_{t}))"]


def expected_agg(e):
    op = e[1:e.index(" ")]
    arg = parse_arg(e)
    node = parse(arg)
    if node[0] == "col" and TABLE[node[1]].full is not None:
        full = TABLE[node[1]].full
        t = TABLE[node[1]].t
        if op == "sum":
            return math.fsum(full.astype(float)), N, math.fsum(np.abs(full.astype(float))), t
        return {"min": full.min(), "max": full.max(), "count": N}[op], N, None, t
    vals, ok, t = reference(arg, TABLE)
    want, n, abs_sum = agg_reference(op, vals, ok, t)
    return want, n, abs_sum, ("u64" if op == "count" else t)


@pytest.mark.parametrize("t", TYPES)
def test_aggregate_sink(env, t):
    exprs = agg_exprs_over_pairs(t) + agg_exprs_over_columns(t)
    for pack in packs(exprs):
        states = run_aggregate(env, pack)
        for e, (dtype, got) in zip(pack, states):
            want, n, abs_sum, rt = expected_agg(e)
            assert dtype == TAG[rt], (e, dtype, rt)
            check_agg_value(e, got, want, n, abs_sum, rt, e[1:e.index(" ")])


def test_aggregate_reference_agrees_with_the_oracle():
    """the closed forms above against the oracle over the full repeated table (one big block: no per-block sum quirk)"""
    exprs = [e for t in TYPES for e in agg_exprs_over_pairs(t) + agg_exprs_over_columns(t) if "col r_" not in e]
    for e in exprs:
        cols = columns_of([e])
        table = {}
        for c in cols:
            col = TABLE[c]
            table[c] = o.Array(TAG[col.t], col.values(), None if col.valid_kind is None else tiled_valid(col))
        try:
            r = o.run_query([e], table=table, is_aggregate=True, worker_threads=1, tail_quirk=False, block_size=1 << 30)
            got = r.columns[0].to_list()[0]
        except o.OracleError as err:
            assert str(err) == "Internal Error: DataValue to array cannot be NONE NULL", (e, str(err))
            got = None
        want, n, abs_sum, rt = expected_agg(e)
        if want is not None and is_float(rt) and not math.isfinite(want):
            # the reference's partial states travel as JSON, where a non-finite float is null: its fold then fails
            assert got is None, (e, got)
            continue
        check_agg_value(e, got, want, n, abs_sum, rt, e[1:e.index(" ")])


# ---------------------------------------------------------------------------------------------
# GROUP BY
# ---------------------------------------------------------------------------------------------
GB_AGGS = ["(sum (col n_i64))", "(min (col n_i64))", "(max (col n_i64))", "(count (col n_i64))", "(sum (col a_f32))",
           "(min (col m_f32))", "(max (col m_f64))"]


def key_id(v, t):
    if v is None:
        return None
    return int(np.asarray(v, NP[t]).view(UINT[t])) if is_float(t) else int(v)


def run_groupby(env, keys, aggs):
    ctx, dev = env
    cols = columns_of(keys + aggs)
    pipe = pipe_for(ctx, aggs, cols, keys=keys)
    groups = pipe.run_groupby(cabi.make_source([dev[c] for c in cols], N), groups_hint=1024)
    kc, kv, lc, lv = pipe.export_groups(groups)
    key_types = [pipe.key_dtype(j) for j in range(len(keys))]
    leaf_types = [pipe.leaf_dtype(k)[0] for k in range(len(aggs))]
    out = {}
    kcols = [(c.to_numpy(groups), None if v is None else v.to_numpy(groups).astype(bool)) for c, v in zip(kc, kv)]
    lcols = [(c.to_numpy(groups), None if v is None else v.to_numpy(groups).astype(bool)) for c, v in zip(lc, lv)]
    for g in range(groups):
        key = []
        for (vals, ok), (kt, _) in zip(kcols, key_types):
            t = next(n for n, tag in TAG.items() if tag == kt)
            key.append(None if ok is not None and not ok[g] else key_id(vals[g], t))
        leaves = [None if ok is not None and not ok[g] else vals[g].item() for vals, ok in lcols]
        assert tuple(key) not in out, f"group {key} exported twice"
        out[tuple(key)] = leaves
    for c in kc + lc + [x for x in kv + lv if x is not None]:
        c.free()
    pipe.destroy()
    return out, key_types, leaf_types


def groupby_reference(keys, aggs):
    key_nodes = [parse(k) for k in keys]
    groups = {}
    for r in range(BLOCK):
        key = []
        for node in key_nodes:
            v, ok, t = evaluate(node, r, TABLE)
            key.append(key_id(v, t) if ok else None)
        groups.setdefault(tuple(key), []).append(r)
    want = {}
    for key, rows in groups.items():
        leaves = []
        for a in aggs:
            op, arg = a[1:a.index(" ")], parse_arg(a)
            vals, ok, t = reference(arg, TABLE)
            leaves.append(agg_reference(op, [vals[r] for r in rows], [ok[r] for r in rows], t) + (t,))
        want[key] = leaves
    return want


def check_groupby(env, keys, aggs):
    got, key_types, leaf_types = run_groupby(env, keys, aggs)
    want = groupby_reference(keys, aggs)
    assert set(got) == set(want), (keys, sorted(set(got) ^ set(want), key=str)[:10])
    for key, leaves in want.items():
        for a, (w, n, abs_sum, t), g in zip(aggs, leaves, got[key]):
            check_agg_value(f"{a} for key {key}", g, w, n, abs_sum, t, a[1:a.index(" ")])
    return got, key_types


@pytest.mark.parametrize("t", TYPES)
def test_groupby_boundary_key(env, t):
    """raw boundary keys: signed narrow keys, -0.0 and 0.0 as two groups, NaN and ±inf keys round-trip by bits"""
    got, key_types = check_groupby(env, [f"(col x_{t})"], GB_AGGS)
    assert key_types == [(TAG[t], False)]
    if is_float(t):
        assert key_id(np.float64(0.0), t) in {k[0] for k in got} and key_id(np.float64(-0.0), t) in {k[0] for k in got}


def test_groupby_key_null_through_a_failed_cast(env):
    keys = ["(+ (col x_u8) (col x_i8))"]                  # coerced to Int8: UInt8 values above 127 give a NULL key
    got, key_types = check_groupby(env, keys, GB_AGGS)
    assert key_types == [(cabi.I8, True)] and (None,) in got


def test_groupby_packed_keys_with_a_nullable_narrow_signed_key_low(env):
    """two keys in one 64-bit word: the nullable Int8 key takes bits 0-7 and its null bit 8, the Int16 key follows"""
    got, key_types = check_groupby(env, ["(col n_i8)", "(col x_i16)"], GB_AGGS)
    assert key_types == [(cabi.I8, True), (cabi.I16, False)]
    got, key_types = check_groupby(env, ["(col x_i8)", "(col n_i16)", "(- (col x_u16) (col x_u8))"], GB_AGGS[:4])
    assert key_types == [(cabi.I8, False), (cabi.I16, True), (cabi.U16, False)]


def test_one_group_matches_the_aggregate_pipe(env):
    """GROUP BY folds f32 sums in double, the aggregate kernel in float: both within the bound of the exact sum"""
    aggs = ["(sum (col r_f32))", "(sum (col a_f32))", "(sum (col r_f64))", "(sum (col a_f64))"]
    got, _, leaf_types = run_groupby(env, ["(col z)"], aggs)
    assert list(got) == [(0,)]
    states = run_aggregate(env, aggs)
    for a, g, (dtype, v) in zip(aggs, got[(0,)], states):
        want, n, abs_sum, t = expected_agg(a)
        check_agg_value(a + " (GROUP BY)", g, want, n, abs_sum, t, "sum")
        check_agg_value(a + " (aggregate)", v, want, n, abs_sum, t, "sum")
    assert leaf_types == [cabi.F32, cabi.F32, cabi.F64, cabi.F64]


# ---------------------------------------------------------------------------------------------
# divide-by-zero errors in every sink
# ---------------------------------------------------------------------------------------------
def run_sink(ctx, sink, expr, cols, dtypes, n):
    names = [f"c{i}" for i in range(len(cols))] + ["k"]
    src = cabi.make_source(cols + [ctx.from_numpy(np.arange(n, dtype=np.uint32))], n)
    kw = dict(columns=names, dtypes=dtypes + [cabi.U32])
    if sink == "map":
        pipe = ctx.pipe([expr], **kw)
    elif sink == "filter":
        pipe = ctx.pipe([expr], predicate="(< (col k) (u32 1000000))", **kw)
    elif sink == "aggregate":
        pipe = ctx.pipe([f"(sum {expr})", f"(count {expr})"], aggregate=True, **kw)
    else:
        pipe = ctx.pipe([f"(sum {expr})", f"(count {expr})"], keys=["(col k)"], **kw)
    try:
        if sink in ("map", "filter"):
            out = ctx.column(pipe.expr_dtype(0), n)
            ov = ctx.column(cabi.BOOL, n) if pipe.expr_nullable(0) else None
            pipe.launch_project(src, [out], n, out_valid=[ov])
            sel, written = pipe.fetch_project()
            assert written == n
            return None if ov is None else ov.to_numpy(n)
        if sink == "aggregate":
            pipe.launch_aggregate(src)
            states, _ = pipe.fetch_aggregate()
            return states
        groups = pipe.run_groupby(src, groups_hint=n)
        assert groups == n
        return groups
    finally:
        pipe.destroy()


@pytest.mark.parametrize("sink", ["map", "filter", "aggregate", "groupby"])
def test_divide_by_zero_in_every_sink(env, sink):
    ctx, _ = env
    n = 1031
    a = np.arange(n, dtype=np.int32) - 500
    # a zero divisor in a valid slot
    b = np.ones(n, np.int32)
    b[777] = 0
    with pytest.raises(cabi.FuseGpuError) as e:
        run_sink(ctx, sink, "(/ (col c0) (col c1))", [ctx.from_numpy(a), ctx.from_numpy(b)], [cabi.I32, cabi.I32], n)
    assert str(e.value) == DIVZERO
    # a divisor that is NULL only because its cast failed: UInt8 200 coerced to Int8 becomes 0 in a NULL slot
    p = (np.arange(n) % 100).astype(np.int8)
    q = np.full(n, 200, np.uint8)
    q[::3] = 7
    res = run_sink(ctx, sink, "(/ (col c0) (col c1))", [ctx.from_numpy(p), ctx.from_numpy(q)], [cabi.I8, cabi.U8], n)
    if sink in ("map", "filter"):
        assert np.array_equal(res, (np.arange(n) % 3 == 0).astype(np.uint8))
    elif sink == "aggregate":
        assert res[0] == (cabi.I8, wrap(sum(int(x) // 7 for x in p[::3]), "i8")) and res[1] == (cabi.U64, n)
    # -0.0 is a zero divisor
    f = np.linspace(-3, 3, n)
    g = np.ones(n)
    g[500] = -0.0
    with pytest.raises(cabi.FuseGpuError) as e:
        run_sink(ctx, sink, "(/ (col c0) (col c1))", [ctx.from_numpy(f), ctx.from_numpy(g)], [cabi.F64, cabi.F64], n)
    assert str(e.value) == DIVZERO


# ---------------------------------------------------------------------------------------------
# SQL literals at the edges of UInt64
# ---------------------------------------------------------------------------------------------
def test_sql_integer_literals_beyond_int64():
    from fuse_query_b200 import _fuse_host as h
    gpu = h.GpuContext.create(0)

    def rows(sql):
        out = []
        for b in h.execute_sql(h.FuseQueryContext.create_ctx(0, gpu), sql):
            cols = [b.column(i).to_list() for i in range(b.num_columns())]
            out += list(zip(*cols)) if cols else []
        return sorted(out)

    n = 1000
    got = rows(f"select number + 9223372036854775807 from system.numbers_mt({n})")    # UInt64: exact
    assert got == [(9223372036854775807 + i,) for i in range(n)] and all(type(r[0]) is int for r in got)
    for lit in ("9223372036854775808", "18446744073709551615"):                         # beyond Int64: Float64
        got = rows(f"select number + {lit} from system.numbers_mt({n})")
        assert got == [(float(i) + float(lit),) for i in range(n)] and all(type(r[0]) is float for r in got)
    huge = "1" + "0" * 399                                                             # a Float64 infinity
    assert rows(f"select number from system.numbers_mt({n}) where number < {huge}") == [(i,) for i in range(n)]
    assert rows(f"select number from system.numbers_mt({n}) where number > {huge}") == []
