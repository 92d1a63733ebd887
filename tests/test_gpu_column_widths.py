"""Fast-field columns at every bit width and splits at every work-unit boundary, through every kernel that reads
them, checked two ways: bit-exact against the CPU oracle (hits, f32 score bits, counts, cells), and against a
brute force over the value arrays this module generated (range-filter hit sets, terms / histogram bucket counts,
min / max, hit order by (value, doc) with None last, exact sums as Python ints). The brute force is what catches
an error the oracle and the kernels share.

Every case names the kernel its batch reaches. The routes follow the dispatch rules of `split_search` in
engine.cu: a batch takes a specialised kernel only when every plan in it qualifies.
  aggscan  match_all, max_hits 0, flat terms / histogram aggregations over always-present columns <= 32 bits,
           no `missing`, at most 4096 cells (agg_kernel.cuh; 32-doc groups, 8192-doc chunks)
  driver   one required term + 0..4 unscored required range / exists filters, no aggregations
           (driver_kernel.cuh; 128-posting blocks, sampled every max(1, blocks / 64)-th block)
  union    an OR of scored terms, top-K by score, no aggregations (union_kernel.cuh; 15360-doc windows)
  window   everything else (kernels.cuh k_window + k_pick + k_select; 16384 / 32768-doc windows), including the
           fast aggregation path (agg_collect_fast / col_raw_doc) when every aggregation reads a FULL column
The aggscan and driver cases assert that the plan fits the rule, so a case cannot drift to another kernel
unnoticed. test_generic_path_agrees re-runs a reduced matrix in a child process with the specialised kernels
switched off and compares it with the oracle and with this process."""
from __future__ import annotations

import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from quickwit_b200 import ffi, plan as P, splitgen as S
from oracle import oracle as O
from helpers import DOC_ASC, DOC_DESC, SCORE_DESC, assert_same, histogram_agg, mapped_to_f64, stats_agg, terms_agg

pytestmark = pytest.mark.gpu

U64 = (1 << 64) - 1
SUM_EXACT_BITS = 40          # QW_SUM_EXACT_BITS
AGGSCAN_MAX_CELLS = 4096     # QA_MAX_CELLS
SMEM_AGG_CELLS = 4096        # QW_SMEM_AGG_CELLS
DRIVER_MAX_FILTERS = 4       # QD_MAX_FILTERS
N_WIDTHS = 20_011            # not a multiple of 32 or 8192: the last group and chunk are partial
MULTI_WIDTHS = (1, 31, 32, 33, 63, 64)
SIZES = (0, 1, 31, 32, 33, 127, 128, 129, 8191, 8192, 8193, 15359, 15360, 15361, 16383, 16385, 32767, 32769, 140_001)
KS = (1, 10, 1000, 4096)


# ---- columns and their brute force --------------------------------------------------------------------------------

class Col:
    """A column as generated: values of doc d are vals[starts[d]:starts[d + 1]] (mapped u64, as Python ints)."""

    def __init__(self, name, ctype, card, starts, vals):
        self.name, self.ctype, self.card = name, ctype, card
        self.starts = [int(x) for x in starts]
        self.vals = [int(x) for x in vals]

    def of(self, d):
        return self.vals[self.starts[d]:self.starts[d + 1]]

    def first(self, d):
        a, b = self.starts[d], self.starts[d + 1]
        return self.vals[a] if a < b else None


def _add(b: S._Builder, cols: dict, name, ctype, card, n, vals, present=None, counts=None):
    vals = np.asarray(vals, dtype=np.uint64)
    if card == ffi.CARD_FULL:
        b.add_column(name, ctype, card, vals, None)
        starts = np.arange(n + 1)
    elif card == ffi.CARD_OPTIONAL:
        b.add_column(name, ctype, card, vals, np.asarray(present, dtype=np.uint32))
        starts = np.zeros(n + 1, dtype=np.int64)
        has = np.zeros(n, dtype=np.int64)
        has[present] = 1
        np.cumsum(has, out=starts[1:])
    else:
        starts = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(counts, out=starts[1:])
        b.add_column(name, ctype, card, vals, starts.astype(np.uint32))
    cols[name] = Col(name, ctype, card, starts, vals)


def _raws(rng, n, bits):
    """n raws spanning exactly [0, 2^bits - 1] (both ends present when n >= 2)."""
    if bits == 0 or n == 0:
        return np.zeros(n, dtype=np.uint64)
    r = rng.integers(0, 1 << 63, size=n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=n, dtype=np.uint64)
    r >>= np.uint64(64 - bits)
    r[0] = 0
    if n > 1:
        r[n // 2] = (1 << bits) - 1
    return r


def _base(bits):
    return 0 if bits == 64 else min(12_345, U64 - ((1 << bits) - 1))


def sum_exact(ctype, bits, num_vals):
    """The rule of qw_col_sum_exact (include/qwgpu_format.h), restated."""
    return ctype != ffi.COL_F64 and bits <= SUM_EXACT_BITS and num_vals * ((1 << bits) - 1) < (1 << 64)


def bf_match(col: Col, lo, hi):
    return [any(lo <= v <= hi for v in col.of(d)) for d in range(len(col.starts) - 1)]


def bf_exists(col: Col):
    return [col.starts[d + 1] > col.starts[d] for d in range(len(col.starts) - 1)]


def bf_order(docs, keys, orders, k):
    """Hit order of a column sort: per key None last, then value in its order; ties by doc id in the first order."""
    def key(d):
        out = []
        for kc, o in zip(keys, orders):
            v = kc.first(d)
            out += [v is None, 0 if v is None else (-v if o == ffi.ORDER_DESC else v)]
        return out + [-d if orders[0] == ffi.ORDER_DESC else d]
    return sorted(docs, key=key)[:k] if k is not None else sorted(docs, key=key)


# ---- aggregation cells --------------------------------------------------------------------------------------------

def _agg_nodes(aggs):
    """(agg, parent index, base cell) in the plan's node order (plan._flatten_aggs), cells laid out node after node."""
    order, pending = [], [(a, -1) for a in aggs]
    while pending:
        a, par = pending.pop(0)
        order.append((a, par))
        me = len(order) - 1
        pending += [(c, me) for c in a.children]
    out, base = [], 0
    for a, par in order:
        mult = 1 if par < 0 else order[par][0].num_buckets
        out.append((a, par, base))
        base += mult * (1 if a.kind == ffi.AGG_STATS else a.num_buckets)
    return out


def _bucket_of(a: P.Agg, col: Col, v):
    if a.kind == ffi.AGG_TERMS:
        return None  # raw index, computed by the caller
    x = mapped_to_f64(col.ctype, v)
    if a.bounds is not None and not (a.bounds[0] <= x <= a.bounds[1]):
        return -1
    pos = math.floor((x - a.offset) / a.interval)
    i = pos - a.base_pos
    return i if 0 <= i < a.num_buckets else -1


def expected_cells(img, cols, aggs, matched):
    """Brute-force cells for flat bucket aggregations (optionally with stats children) and top-level stats.
    Stats cells are (count, raw_sum, min_mapped, max_mapped, typed_sum, sum of |value|) with Python-int sums."""
    nodes = _agg_nodes(aggs)
    total = sum(1 if a.kind == ffi.AGG_STATS else a.num_buckets for a, par, _ in nodes if par < 0)
    total += sum(nodes[par][0].num_buckets for a, par, _ in nodes if par >= 0)
    icols = img.columns()
    names = img.column_names()
    exp = {}
    for a, par, base in nodes:
        if par >= 0:
            continue
        col = cols[names[a.column]]
        ic = icols[a.column]
        if a.kind == ffi.AGG_STATS:
            exp[base] = _stats([v for d in matched for v in col.of(d)], ic, col.ctype)
            continue
        counts = [0] * a.num_buckets
        members = [[] for _ in range(a.num_buckets)]
        for d in matched:
            for v in col.of(d):
                bk = (v - ic.min_value) // ic.gcd if a.kind == ffi.AGG_TERMS else _bucket_of(a, col, v)
                if bk >= 0:
                    counts[bk] += 1
                    members[bk].append(d)
        for i, c in enumerate(counts):
            exp[base + i] = c
        for ch in a.children:
            cbase = next(bb for aa, pp, bb in nodes if aa is ch)
            ccol, cic = cols[names[ch.column]], icols[ch.column]
            for i in range(a.num_buckets):
                exp[cbase + i] = _stats([v for d in members[i] for v in ccol.of(d)], cic, ccol.ctype)
    return exp, total


def _stats(vals, ic, ctype):
    if not vals:
        return (0,)
    raws = [(v - ic.min_value) // ic.gcd for v in vals]
    if ctype in (ffi.COL_I64, ffi.COL_DATETIME):
        typed = sum(S.u64_to_i64(v) for v in vals)
    elif ctype == ffi.COL_F64:
        typed = math.fsum(S.u64_to_f64(v) for v in vals)
    else:
        typed = sum(vals)
    return (len(vals), sum(raws), min(vals), max(vals), typed, sum(abs(mapped_to_f64(ctype, v)) for v in vals))


def f64_cells(img, aggs):
    """Cells whose sum is an f64 sum (accumulated in another order on the device: compared within a bound)."""
    out = []
    icols = img.columns()
    nodes = _agg_nodes(aggs)
    for a, par, base in nodes:
        if a.kind != ffi.AGG_STATS or a.column == ffi.ABSENT:
            continue
        ic = icols[a.column]
        if not sum_exact(ic.type, ic.bits, ic.num_vals):
            out += list(range(base, base + (1 if par < 0 else nodes[par][0].num_buckets)))
    return out


def check_cells(got_cells, img, cols, aggs, matched, ctx):
    exp, total = expected_cells(img, cols, aggs, matched)
    assert len(got_cells) == total, f"{ctx}: {len(got_cells)} cells, expected {total}"
    icols = img.columns()
    stats_cols = {base: icols[a.column] for a, par, base in _agg_nodes(aggs) if a.kind == ffi.AGG_STATS}
    for i, e in exp.items():
        g = got_cells[i]
        if isinstance(e, int):
            assert g[0] == e, f"{ctx}: bucket cell {i}: count {g[0]}, brute force {e}"
            continue
        assert g[0] == e[0], f"{ctx}: stats cell {i}: count {g[0]}, brute force {e[0]}"
        if not e[0]:
            continue
        cnt, raw_sum, mn, mx, typed, abs_sum = e
        assert (g[2], g[3]) == (mn, mx), f"{ctx}: stats cell {i}: min/max {g[2:]} != {(mn, mx)}"
        ic = stats_cols[max(b for b in stats_cols if b <= i)]  # the stats node that owns cell i
        if sum_exact(ic.type, ic.bits, ic.num_vals):
            assert raw_sum < (1 << 64)
            assert g[1] == raw_sum, f"{ctx}: stats cell {i}: exact raw sum {g[1]} != {raw_sum}"
        else:
            s = S.struct.unpack("<d", S.struct.pack("<Q", g[1]))[0]
            assert abs(s - typed) <= cnt * 2.0 ** -52 * abs_sum + 1e-300, f"{ctx}: stats cell {i}: f64 sum {s!r} vs {typed}"


# ---- splits -------------------------------------------------------------------------------------------------------

def widths_split(split_id="widths-0", n=N_WIDTHS, seed=1):
    """Every width 0..64 as FULL u64 (shuffled `u{b}` and doc-ordered `s{b}`), a gcd > 1 column, negative i64, f64,
    datetime, OPTIONAL `o{b}` / MULTI `m{b}` at widths 1, 31, 32, 33, 63, 64. Terms: `every`, `half`, `rare`."""
    rng = np.random.default_rng(seed)
    b = S._Builder(n)
    cols = {}
    body = b.add_field("body", 0, ffi.TOK_RAW, None, n)
    b.add_term(body, b"every", np.arange(n, dtype=np.uint32), None)
    half = np.sort(rng.choice(n, n // 2, replace=False)).astype(np.uint32)
    b.add_term(body, b"half", half, None)
    b.add_term(body, b"rare", np.array([0, 31, 32, 8191, 8192, n - 1], dtype=np.uint32), None)
    for bits in range(65):
        raws = _raws(rng, n, bits)
        _add(b, cols, f"u{bits}", ffi.COL_U64, ffi.CARD_FULL, n, raws + np.uint64(_base(bits)))
        _add(b, cols, f"s{bits}", ffi.COL_U64, ffi.CARD_FULL, n, np.sort(raws) + np.uint64(_base(bits)))
    _add(b, cols, "gcd", ffi.COL_U64, ffi.CARD_FULL, n, 7 + 1000 * rng.integers(0, 5000, n, dtype=np.uint64))
    for bits in (7, 33, 63, 64):  # i64 around and below zero; 64 bits covers i64::MIN .. i64::MAX
        lo = -(1 << (bits - 1))
        _add(b, cols, f"i{bits}", ffi.COL_I64, ffi.CARD_FULL, n,
             [S.i64_to_u64(lo + int(r)) for r in _raws(rng, n, bits)])
    _add(b, cols, "f_small", ffi.COL_F64, ffi.CARD_FULL, n, [S.f64_to_u64(float(x)) for x in rng.normal(0, 1e3, n)])
    _add(b, cols, "f_wide", ffi.COL_F64, ffi.CARD_FULL, n,
         [S.f64_to_u64(float(x)) for x in rng.choice([-1, 1], n) * 10.0 ** rng.uniform(-300, 300, n)])
    for bits in (20, 45):
        _add(b, cols, f"dt{bits}", ffi.COL_DATETIME, ffi.CARD_FULL, n,
             [S.i64_to_u64(1_700_000_000 * 10**9 + 1000 * int(r)) for r in _raws(rng, n, bits)])
    present = np.array([d for d in range(n) if d % 3], dtype=np.int64)
    counts = np.array([d % 4 for d in range(n)], dtype=np.int64)
    for bits in MULTI_WIDTHS:
        _add(b, cols, f"o{bits}", ffi.COL_U64, ffi.CARD_OPTIONAL, n, _raws(rng, len(present), bits) + np.uint64(_base(bits)), present=present)
        _add(b, cols, f"m{bits}", ffi.COL_U64, ffi.CARD_MULTI, n, _raws(rng, int(counts.sum()), bits) + np.uint64(_base(bits)), counts=counts)
    img = b.finish(split_id)
    post = {"every": list(range(n)), "half": [int(d) for d in half]}
    icols = img.columns()
    for bits in range(65):
        assert icols[img.column_ord(f"u{bits}")].bits == bits and icols[img.column_ord(f"s{bits}")].bits == bits
    for bits in MULTI_WIDTHS:
        assert icols[img.column_ord(f"o{bits}")].bits == bits and icols[img.column_ord(f"m{bits}")].bits == bits
    assert icols[img.column_ord("gcd")].gcd == 1000
    return img, cols, post


def sized_split(n, split_id, seed=2):
    """n docs; terms: `every` doc, exactly 128 and 129 docs, one posting at the last doc, a sparse term, a random half.
    Columns: `ts` (doc order), `val` (shuffled 20-bit), `code` (5 values)."""
    rng = np.random.default_rng(seed + n)
    b = S._Builder(n)
    cols, post = {}, {}
    lengths = (1 + (np.arange(n) * 7919) % 40).astype(np.uint32)
    L = ffi.img_lib()
    fn = np.array([L.qwgpu_fieldnorm_to_id(int(x)) for x in lengths[:4096]], dtype=np.uint8)
    fn = np.resize(fn, n) if n else np.zeros(0, dtype=np.uint8)
    body = b.add_field("body", ffi.FIELD_HAS_FREQS | ffi.FIELD_HAS_FIELDNORMS, ffi.TOK_DEFAULT, fn, int(lengths.sum()))
    if n:
        post["every"] = np.arange(n)
        post["last"] = np.array([n - 1])
        post["sparse"] = np.arange(n // 2 % 97, n, 97)
        post["half"] = np.sort(rng.choice(n, max(1, n // 2), replace=False))
    if n >= 128:
        post["t128"] = np.sort(rng.choice(n, 128, replace=False))
    if n >= 129:
        post["t129"] = np.sort(rng.choice(n, 129, replace=False))
    for t, docs in sorted(post.items()):
        docs = docs.astype(np.uint32)
        b.add_term(body, t.encode(), docs, (1 + (docs * 31) % 3).astype(np.uint32))
    _add(b, cols, "ts", ffi.COL_U64, ffi.CARD_FULL, n, 1_000_000 + np.arange(n, dtype=np.uint64) // 3)
    _add(b, cols, "val", ffi.COL_U64, ffi.CARD_FULL, n, _raws(rng, n, 20))
    _add(b, cols, "code", ffi.COL_U64, ffi.CARD_FULL, n, (np.arange(n, dtype=np.uint64) * 7) % 5)
    return b.finish(split_id), cols, {t: [int(x) for x in d] for t, d in post.items()}


# ---- dispatch rules (engine.cu split_search) ----------------------------------------------------------------------

def fits_aggscan(img, root, max_hits, aggs):
    icols = img.columns()
    if root.kind != ffi.NODE_ALL or max_hits != 0 or not aggs:
        return False
    cells = sum(a.num_buckets for a in aggs)
    return cells <= AGGSCAN_MAX_CELLS and all(
        not a.children and a.kind in (ffi.AGG_TERMS, ffi.AGG_HISTOGRAM) and a.missing is None and a.column != ffi.ABSENT
        and icols[a.column].cardinality == ffi.CARD_FULL and icols[a.column].bits <= 32 and 0 < a.num_buckets <= SMEM_AGG_CELLS
        for a in aggs)


def fits_driver(root, aggs):
    if aggs or root.kind != ffi.NODE_BOOL or not root.children:
        return False
    t, filters = root.children[0], root.children[1:]
    return (t.kind == ffi.NODE_TERM and t.occur in (ffi.OCCUR_MUST, ffi.OCCUR_FILTER) and len(filters) <= DRIVER_MAX_FILTERS
            and all(f.kind in (ffi.NODE_RANGE, ffi.NODE_EXISTS) and f.occur == ffi.OCCUR_FILTER for f in filters))


# ---- running a case -----------------------------------------------------------------------------------------------

class Case:
    """One plan over one split plus what the brute force expects of it."""

    def __init__(self, name, route, split, root, k, sort, aggs=(), sa=None, matched=None, order_keys=None):
        img, cols, _ = split
        self.name, self.route, self.split = f"[{route}] {name} ({img.split_id})", route, split
        self.root, self.k, self.sort, self.aggs, self.matched, self.order_keys = root, k, sort, list(aggs), matched, order_keys
        self.plan = P.make_plan(root, k, sort, aggs=self.aggs, search_after=sa)
        if route == "aggscan":
            assert fits_aggscan(img, root, k, self.aggs), self.name
        if route == "driver":
            assert fits_driver(root, self.aggs), self.name


def run_batch(ctx, cases):
    """One split_search call over the cases' splits; every result against the oracle and the brute force."""
    got = ctx.split_search([c.split[0].split_id for c in cases], [c.plan for c in cases])
    for c, g in zip(cases, got):
        img, cols, _ = c.split
        want = O.split_search(img, c.plan)
        assert_same(g, want, f64_sum_cells=f64_cells(img, c.aggs), ctx=c.name)
        check_brute(c, g)
    return got


def check_brute(c: Case, r):
    img, cols, _ = c.split
    if c.matched is None:
        return
    m = c.matched
    assert r.num_hits == len(m), f"{c.name}: {r.num_hits} hits, brute force {len(m)}"
    if c.aggs:
        check_cells(r.cells, img, cols, c.aggs, m, c.name)
    if c.k and c.order_keys is not None:
        keys, orders = c.order_keys
        if keys:
            want = bf_order(m, keys, orders, None)
        else:
            want = sorted(m, reverse=orders[0] == ffi.ORDER_DESC)
        want = want[:c.k]
        assert [h[0] for h in r.hits] == want, f"{c.name}: hit order differs from the brute force"
        for h in r.hits:
            for i, kc in enumerate(keys):
                v = kc.first(h[0])
                assert bool(h[1] >> i & 1) == (v is not None) and (v is None or h[2 + i] == v), f"{c.name}: sort value of doc {h[0]}"
    elif c.k:
        assert len(r.hits) == min(c.k, len(m)), c.name


def col_sort(img, name, order):
    c = img.column_ord(name)
    return (ffi.SORT_COLUMN, order, c if c >= 0 else ffi.ABSENT)


def _hist(img, cols, name, parts=37.3, offset=0.0, bounds=None, children=()):
    ic = img.columns()[img.column_ord(name)]
    lo, hi = mapped_to_f64(ic.type, ic.min_value), mapped_to_f64(ic.type, ic.max_value)
    interval = max((hi - lo) / parts, 1.0) if ic.type != ffi.COL_F64 else (hi - lo) / parts
    if bounds is not None:
        bounds = (lo + (hi - lo) * bounds[0], lo + (hi - lo) * bounds[1])
    return histogram_agg(img, name, interval, offset=offset * interval, bounds=bounds, children=children)


# ---- Part A: column widths ----------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def wsplit(gpu_ctx):
    sp = widths_split()
    gpu_ctx.register_split(sp[0])
    yield sp
    gpu_ctx.unregister_split(sp[0].split_id)


def aggscan_cases(sp, widths=range(33)):
    img, cols, _ = sp
    out = []
    every = list(range(img.num_docs))
    for bits in widths:
        for name in (f"u{bits}", f"s{bits}"):
            aggs = [_hist(img, cols, name), _hist(img, cols, name, parts=5.5, offset=0.3, bounds=(0.2, 0.7))]
            if bits <= 10:
                aggs.append(terms_agg(img, name))
            out.append(Case(f"{name}: histograms + terms", "aggscan", sp, P.match_all(), 0, DOC_DESC, aggs, matched=every))
    return out


def test_aggscan_every_width_to_32(gpu_ctx, wsplit):
    """Widths 0..32 shuffled and doc-ordered (bucket cache / group min-max shortcut vs the straddle path), terms at
    1, 2 and >= 3 bits, histograms whose buckets straddle 32-doc groups, hard bounds, a partial last group / chunk."""
    for c in aggscan_cases(wsplit):
        run_batch(gpu_ctx, [c])


def window_agg_cases(sp, widths=range(65)):
    img, cols, post = sp
    half = post["half"]
    out = []
    for bits in widths:
        for name in (f"u{bits}", f"s{bits}"):
            # fast path: bucket nodes with stats children and a top-level stats node, all over FULL columns
            aggs = [terms_agg(img, "u3", children=[stats_agg(img, name)]), _hist(img, cols, name, children=[stats_agg(img, "u41")]),
                    stats_agg(img, name)]
            out.append(Case(f"{name}: term root, stats children", "window", sp, P.term(img, "body", "half"), 0, DOC_DESC, aggs, matched=half))
    return out


def test_window_fast_aggregations_every_width(gpu_ctx, wsplit):
    """agg_collect_fast / col_raw_doc at widths 0..64 (the 32-bit funnel-shift path, 64-bit loads, values crossing
    words), stats at 40 / 41 bits (exact integer / f64 sum switch)."""
    for c in window_agg_cases(wsplit):
        run_batch(gpu_ctx, [c])


def test_window_generic_aggregations_optional_multi_typed(gpu_ctx, wsplit):
    img, cols, post = wsplit
    half = post["half"]
    every = list(range(img.num_docs))
    names = [f"o{b}" for b in MULTI_WIDTHS] + [f"m{b}" for b in MULTI_WIDTHS] + ["gcd", "i7", "i33", "i63", "i64", "f_small", "f_wide", "dt20", "dt45"]
    for name in names:
        for root, m in ((P.term(img, "body", "half"), half), (P.match_all(), every)):
            aggs = [_hist(img, cols, name, children=[stats_agg(img, name)]), stats_agg(img, name)]
            run_batch(gpu_ctx, [Case(f"{name}: histogram + stats", "window", wsplit, root, 0, DOC_DESC, aggs, matched=m)])
    for name in ("m1", "o1", "gcd"):
        run_batch(gpu_ctx, [Case(f"{name}: terms", "window", wsplit, P.match_all(), 0, DOC_DESC, [terms_agg(img, name)], matched=every)])
    for name in ("gcd", "i7", "dt20"):  # FULL typed columns <= 32 bits reach aggscan too
        ic = img.columns()[img.column_ord(name)]
        if ic.bits <= 32:
            run_batch(gpu_ctx, [Case(f"{name}: histogram", "aggscan", wsplit, P.match_all(), 0, DOC_DESC, [_hist(img, cols, name)], matched=every)])


def driver_cases(sp, names):
    img, cols, _ = sp
    every = list(range(img.num_docs))
    out = []
    for name in names:
        col, ic = cols[name], img.columns()[img.column_ord(name)]
        lo, hi = ic.min_value, ic.max_value
        mid = sorted(col.vals)[len(col.vals) // 2] if col.vals else lo
        bounds = [(lo, hi), (lo, lo), (hi, hi), (mid, hi), (lo, mid)]
        if hi - lo >= 2:
            bounds.append((lo + 1, hi - 1))
        for blo, bhi in bounds:
            root = P.bool_([P.term(img, "body", "every"), P.range_(img, name, blo, bhi)])
            m = [d for d, ok in enumerate(bf_match(col, blo, bhi)) if ok]
            sort, keys = ([col_sort(img, name, ffi.ORDER_ASC)], ([col], [ffi.ORDER_ASC])) if col.card != ffi.CARD_MULTI else (DOC_DESC, ([], [ffi.ORDER_DESC]))
            out.append(Case(f"{name} in [{blo}, {bhi}]", "driver", sp, root, 100, sort, matched=m, order_keys=keys))
        root = P.bool_([P.term(img, "body", "every"), P.exists(img, name, occur=ffi.OCCUR_FILTER)])
        m = [d for d, ok in enumerate(bf_exists(col)) if ok]
        out.append(Case(f"exists {name}", "driver", sp, root, 10, DOC_DESC, matched=m, order_keys=([], [ffi.ORDER_DESC])))
    return out


def test_driver_range_filters_every_width(gpu_ctx, wsplit):
    img, cols, _ = wsplit
    names = [f"u{b}" for b in range(65)] + [f"s{b}" for b in (1, 32, 33, 64)] + [f"o{b}" for b in MULTI_WIDTHS] + \
            [f"m{b}" for b in MULTI_WIDTHS] + ["gcd", "i7", "i33", "i63", "i64", "f_small", "f_wide", "dt20", "dt45"]
    for c in driver_cases(wsplit, names):
        run_batch(gpu_ctx, [c])
    # four filters at once (different widths, one multi-valued), and a range over a column the split lacks
    c3, c33, c64, m31 = cols["u3"], cols["u33"], cols["u64"], cols["m31"]
    ic = {k: img.columns()[img.column_ord(k)] for k in ("u3", "u33", "u64", "m31")}
    f = [("u3", 1 + ic["u3"].min_value, 6 + ic["u3"].min_value), ("u33", ic["u33"].min_value, ic["u33"].min_value + (1 << 32)),
         ("u64", 1 << 62, U64), ("m31", ic["m31"].min_value, ic["m31"].min_value + (1 << 30))]
    root = P.bool_([P.term(img, "body", "every")] + [P.range_(img, n, lo, hi) for n, lo, hi in f])
    m = [d for d in range(img.num_docs) if all(any(lo <= v <= hi for v in cols[n].of(d)) for n, lo, hi in f)]
    run_batch(gpu_ctx, [Case("four filters", "driver", wsplit, root, 1000, DOC_ASC, matched=m, order_keys=([], [ffi.ORDER_ASC]))])
    root = P.bool_([P.term(img, "body", "every"), P.range_(img, "no_such_column", 0, U64)])
    run_batch(gpu_ctx, [Case("absent column", "driver", wsplit, root, 10, DOC_DESC, matched=[], order_keys=([], [ffi.ORDER_DESC]))])


KEY_PAIRS = [(b1, b2) for b1 in (1, 17, 31, 32, 33, 47, 48, 49, 63, 64) for b2 in (0, 1, 15, 16, 33, 48, 63, 64)]


def sort_cases(sp, pairs=KEY_PAIRS, ks=(1, 1000)):
    """Two-column sorts whose [has1][r1][has2][r2][doc'] fields cross each 64-bit word boundary of the 192-bit key."""
    img, cols, _ = sp
    every = list(range(img.num_docs))
    out = []
    for i, (b1, b2) in enumerate(pairs):
        o1, o2 = (ffi.ORDER_DESC, ffi.ORDER_ASC) if i % 2 else (ffi.ORDER_ASC, ffi.ORDER_DESC)
        c1, c2 = cols[f"u{b1}"], cols[f"u{b2}"]
        sort = [col_sort(img, c1.name, o1), col_sort(img, c2.name, o2)]
        for k in ks:
            out.append(Case(f"sort u{b1} {o1} u{b2} {o2} k={k}", "window", sp, P.match_all(), k, sort, matched=every,
                            order_keys=([c1, c2], [o1, o2])))
    return out


def test_composite_keys_across_word_boundaries(gpu_ctx, wsplit):
    img, cols, _ = wsplit
    for c in sort_cases(wsplit):
        run_batch(gpu_ctx, [c])
    # an optional first key (has-value bit, None last) and a negative i64 second key
    for o in (ffi.ORDER_ASC, ffi.ORDER_DESC):
        sort = [col_sort(img, "o33", o), col_sort(img, "i63", 1 - o)]
        run_batch(gpu_ctx, [Case(f"sort o33/i63 {o}", "window", wsplit, P.match_all(), 500, sort, matched=list(range(img.num_docs)),
                                 order_keys=([cols["o33"], cols["i63"]], [o, 1 - o]))])


def test_search_after_on_wide_keys(gpu_ctx, wsplit):
    img, cols, _ = wsplit
    every = list(range(img.num_docs))
    for b1, b2 in ((64, 64), (33, 48), (63, 1), (17, 0), (1, 63)):
        for o1, o2 in ((ffi.ORDER_ASC, ffi.ORDER_DESC), (ffi.ORDER_DESC, ffi.ORDER_ASC)):
            c1, c2 = cols[f"u{b1}"], cols[f"u{b2}"]
            order = bf_order(every, [c1, c2], [o1, o2], None)
            for at in (0, 37, len(order) // 2):
                d = order[at]
                sa = ffi.QwSearchAfter(present=1, has_v1=1, has_v2=1, compare_on_equal=1, precomp_order=0, doc_id=d,
                                       v1=c1.first(d), v2=c2.first(d))
                c = Case(f"search_after u{b1}/u{b2} from #{at}", "window", wsplit, P.match_all(), 300,
                         [col_sort(img, c1.name, o1), col_sort(img, c2.name, o2)], sa=sa, matched=every, order_keys=([c1, c2], [o1, o2]))
                got = run_batch_sa(gpu_ctx, c)
                assert [h[0] for h in got.hits] == order[at + 1: at + 301], c.name


def run_batch_sa(ctx, c):
    # search_after: hits are the ones strictly after the given position; num_hits still counts every match
    g = ctx.split_search([c.split[0].split_id], [c.plan])[0]
    assert_same(g, O.split_search(c.split[0], c.plan), ctx=c.name)
    assert g.num_hits == len(c.matched)
    return g


@pytest.fixture(scope="module")
def other_splits(gpu_ctx):
    """A second widths split (other seed) and an empty split with the same columns."""
    sp = widths_split("widths-1", n=9_001, seed=9)
    b = S._Builder(0)
    cols = {}
    for name in ("u3", "u17", "u32", "u41"):
        _add(b, cols, name, ffi.COL_U64, ffi.CARD_FULL, 0, np.zeros(0, dtype=np.uint64))
    empty = (b.finish("empty-0"), cols, {})
    for s in (sp, empty):
        gpu_ctx.register_split(s[0])
    yield sp, empty
    for s in (sp, empty):
        gpu_ctx.unregister_split(s[0].split_id)


def test_mixed_batch_with_an_empty_split(gpu_ctx, wsplit, other_splits):
    """One split_search over several splits: one aggregation reads columns of different widths (the aggscan slots
    are sized by the widest), one split is empty; the same for the driver and union shapes."""
    sp1, empty = other_splits
    img0, img1, imge = wsplit[0], sp1[0], empty[0]
    cases = []
    for sp, names in ((wsplit, ("u3", "u17", "u32")), (sp1, ("u32", "u3", "u17")), (wsplit, ("s1", "s31", "s2"))):
        img = sp[0]
        aggs = [terms_agg(img, names[0]) if names[0] in ("u3", "s1") else _hist(img, sp[1], names[0]), _hist(img, sp[1], names[1]),
                _hist(img, sp[1], names[2], parts=3.1)]
        cases.append(Case(f"widths {names}", "aggscan", sp, P.match_all(), 0, DOC_DESC, aggs, matched=list(range(img.num_docs))))
    cases.append(Case("empty", "aggscan", empty, P.match_all(), 0, DOC_DESC, [terms_agg(imge, "u3")], matched=[]))
    run_batch(gpu_ctx, cases)
    # window fast aggregations with 40 / 41-bit stats, one empty split
    cases = [Case("stats 40/41", "window", sp, P.term(sp[0], "body", "every"), 0, DOC_DESC,
                  [terms_agg(sp[0], "u3", children=[stats_agg(sp[0], "u40")]), stats_agg(sp[0], "u41")], matched=list(range(sp[0].num_docs)))
             for sp in (wsplit, sp1)]
    cases.append(Case("empty", "window", empty, P.match_all(), 0, DOC_DESC, [terms_agg(imge, "u3", children=[stats_agg(imge, "u41")])], matched=[]))
    run_batch(gpu_ctx, cases)
    for route, mk in (("driver", lambda img: P.bool_([P.term(img, "body", "every"), P.exists(img, "u17", occur=ffi.OCCUR_FILTER)])),
                      ("union", lambda img: P.bool_([P.term(img, "body", t, occur=ffi.OCCUR_SHOULD) for t in ("rare", "half")]))):
        cases = [Case(f"{route} + empty", route, sp, mk(sp[0]), 50, SCORE_DESC if route == "union" else DOC_DESC) for sp in (wsplit, empty, sp1)]
        run_batch(gpu_ctx, cases)


# ---- Part B: split sizes at the kernels' work units ---------------------------------------------------------------

@pytest.fixture(scope="module")
def sized(gpu_ctx):
    sps = [sized_split(n, f"size-{n}") for n in SIZES]
    for sp in sps:
        gpu_ctx.register_split(sp[0])
    yield sps
    for sp in sps:
        gpu_ctx.unregister_split(sp[0].split_id)


def size_cases(sp, k):
    img, cols, post = sp
    n = img.num_docs
    terms = [t for t in ("every", "t128", "t129", "last", "sparse") if t in post]
    out = []
    # union: OR of scored terms, top-K by score (the oracle checks the scores; the brute force the hit count)
    root = P.bool_([P.term(img, "body", t, occur=ffi.OCCUR_SHOULD) for t in terms] or [P.term(img, "body", "every", occur=ffi.OCCUR_SHOULD)])
    out.append(Case(f"OR {terms} k={k}", "union", sp, root, k, SCORE_DESC, matched=sorted({d for t in terms for d in post[t]})))
    # driver: term + range filter, sorted by a column
    val = cols["val"]
    lo, hi = (1 << 18), (3 << 18)
    root = P.bool_([P.term(img, "body", "every"), P.range_(img, "val", lo, hi)])
    m = [d for d, ok in enumerate(bf_match(val, lo, hi)) if ok and "every" in post]
    out.append(Case(f"every + val range k={k}", "driver", sp, root, k, [col_sort(img, "ts", ffi.ORDER_DESC)], matched=m,
                    order_keys=([cols["ts"]], [ffi.ORDER_DESC])))
    # window: a nested bool with must_not
    inner = P.bool_([P.term(img, "body", "t129", occur=ffi.OCCUR_SHOULD), P.term(img, "body", "last", occur=ffi.OCCUR_SHOULD)], occur=ffi.OCCUR_SHOULD)
    root = P.bool_([P.term(img, "body", "every"), P.term(img, "body", "sparse", occur=ffi.OCCUR_MUST_NOT), inner])
    m = sorted(set(post.get("every", [])) - set(post.get("sparse", [])))
    out.append(Case(f"every -sparse (t129 | last) k={k}", "window", sp, root, k, [col_sort(img, "val", ffi.ORDER_ASC)], matched=m,
                    order_keys=([val], [ffi.ORDER_ASC])))
    return out


def size_agg_case(sp):
    img, cols, _ = sp
    if img.num_docs == 0:
        # an empty split has no value range to build a histogram over
        return Case("terms", "aggscan", sp, P.match_all(), 0, DOC_DESC, [terms_agg(img, "code")], matched=[])
    return Case("terms + histogram", "aggscan", sp, P.match_all(), 0, DOC_DESC, [terms_agg(img, "code"), _hist(img, cols, "val", parts=100.5)],
                matched=list(range(img.num_docs)))


def test_split_sizes_alone(gpu_ctx, sized):
    for sp in sized:
        run_batch(gpu_ctx, [size_agg_case(sp)])
        for k in KS:
            for c in size_cases(sp, k):
                run_batch(gpu_ctx, [c])


def test_split_sizes_together(gpu_ctx, sized):
    run_batch(gpu_ctx, [size_agg_case(sp) for sp in sized])
    for k in KS:
        for i in range(3):
            run_batch(gpu_ctx, [size_cases(sp, k)[i] for sp in sized])


# ---- Part C: stats sums beyond 2^64 -------------------------------------------------------------------------------

def test_stats_sums_beyond_the_exact_limit(gpu_ctx):
    """40-bit raws whose sum passes 2^64: 18 M values of a multi-valued column (generic agg_stats) and a FULL column of
    2^24 + 2^20 docs (privatised stat_update of the fast path). Both must take the f64 sum; the finished sum is
    within the f64 accumulation bound of the exact Python-int sum."""
    rng = np.random.default_rng(7)
    n_multi, per_doc, n_full = 3_000_000, 6, (1 << 24) + (1 << 20)
    mv = (1 << 40) - 1 - rng.integers(0, 1 << 20, size=n_multi * per_doc, dtype=np.uint64)
    mv[0] = 0
    fv = (1 << 40) - 1 - rng.integers(0, 1 << 20, size=n_full, dtype=np.uint64)
    fv[1] = 0
    b = S._Builder(n_multi)
    b.add_column("v", ffi.COL_U64, ffi.CARD_MULTI, mv, np.arange(0, n_multi * per_doc + 1, per_doc, dtype=np.uint32))
    multi = b.finish("sum-multi")
    b = S._Builder(n_full)
    b.add_column("v", ffi.COL_U64, ffi.CARD_FULL, fv, None)
    full = b.finish("sum-full")

    def exact(v):
        return (int((v >> np.uint64(20)).sum(dtype=np.uint64)) << 20) + int((v & np.uint64((1 << 20) - 1)).sum(dtype=np.uint64))

    for img, vals in ((multi, mv), (full, fv)):
        ic = img.columns()[0]
        assert ic.bits == 40 and not sum_exact(ic.type, ic.bits, ic.num_vals)
        gpu_ctx.register_split(img)
        try:
            plan = P.make_plan(P.match_all(), 0, DOC_DESC, aggs=[stats_agg(img, "v")])
            got = gpu_ctx.split_search([img.split_id], [plan])[0]
            assert_same(got, O.split_search(img, plan), f64_sum_cells=[0], ctx=img.split_id)
            s = S.struct.unpack("<d", S.struct.pack("<Q", got.cells[0][1]))[0]
            e = exact(vals)
            assert e >= 1 << 64
            assert got.cells[0][0] == len(vals) and got.cells[0][2:] == (0, int(vals.max()))
            assert abs(s - e) <= len(vals) * 2.0 ** -52 * e, f"{img.split_id}: sum {s!r} vs exact {e}"
        finally:
            gpu_ctx.unregister_split(img.split_id)


# ---- Part D: the same matrix through the generic path -------------------------------------------------------------

GENERIC_ENV = {"QWGPU_OLD_AGGS": "1", "QWGPU_NO_DRIVER": "1", "QWGPU_OLD_UNION": "1", "QWGPU_DYNAMIC_WORK": "1", "QWGPU_STRIDE_CAP": "4"}


def reduced_matrix():
    """Batches (lists of cases) of a reduced A + B matrix; the splits are rebuilt from their seeds in each process
    (under ids of their own, so that they never replace the module's registered splits)."""
    wsp = widths_split("matrix-widths-0")
    sized_sps = [sized_split(n, f"matrix-size-{n}") for n in (0, 31, 33, 128, 8193, 15361, 16385, 32769, 140_001)]
    batches = [[c] for c in aggscan_cases(wsp, widths=(0, 1, 2, 3, 7, 16, 31, 32))]
    batches += [[c] for c in window_agg_cases(wsp, widths=(0, 1, 32, 33, 40, 41, 63, 64))]
    batches += [[c] for c in driver_cases(wsp, ["u1", "u32", "u33", "u64", "o33", "m63", "i64", "f_wide"])]
    batches += [[c] for c in sort_cases(wsp, pairs=[(64, 64), (63, 1), (33, 48), (1, 0)], ks=(10,))]
    batches.append([size_agg_case(sp) for sp in sized_sps])
    for k in (1, 1000, 4096):
        for i in range(3):
            batches.append([size_cases(sp, k)[i] for sp in sized_sps])
    return [wsp] + sized_sps, batches


def _run_matrix(ctx):
    splits, batches = reduced_matrix()
    for sp in splits:
        ctx.register_split(sp[0])
    try:
        out = []
        for batch in batches:
            out.append([(g.num_hits, [list(h) for h in g.hits], [list(c) for c in g.cells]) for g in run_batch(ctx, batch)])
        return out
    finally:
        for sp in splits:
            ctx.unregister_split(sp[0].split_id)


def _child_main(out_path):
    from quickwit_b200.service import SearcherContext
    ctx = SearcherContext(0)
    try:
        res = _run_matrix(ctx)
    finally:
        ctx.close()
    with open(out_path, "w") as f:
        json.dump(res, f)


def test_generic_path_agrees(gpu_ctx, tmp_path):
    """The A/B switches and QWGPU_DYNAMIC_WORK / QWGPU_STRIDE_CAP are read once per process, so the reduced matrix
    runs again in a child process with them set. The child checks every result against the oracle and the brute
    force itself; here its results must equal this process's."""
    mine = _run_matrix(gpu_ctx)
    out = tmp_path / "generic.json"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, **GENERIC_ENV)
    env["PYTHONPATH"] = os.pathsep.join([root, os.path.join(root, "tests")] + ([env["PYTHONPATH"]] if env.get("PYTHONPATH") else []))
    code = f"import test_gpu_column_widths as T; T._child_main({str(out)!r})"
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"generic-path child failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    theirs = json.loads(out.read_text())
    _, batches = reduced_matrix()
    assert len(theirs) == len(mine) == len(batches)
    for batch, a, b in zip(batches, mine, theirs):
        for c, x, y in zip(batch, a, b):
            f64 = set(f64_cells(c.split[0], c.aggs))
            assert x[0] == y[0] and x[1] == y[1], f"{c.name}: hits differ between the specialised and the generic path"
            for i, (p, q) in enumerate(zip(x[2], y[2])):
                if i in f64:
                    fa, fb = (S.struct.unpack("<d", S.struct.pack("<Q", v))[0] for v in (p[1], q[1]))
                    assert p[0] == q[0] and p[2:] == q[2:] and abs(fa - fb) <= 1e-9 * max(1.0, abs(fb)), f"{c.name}: cell {i}"
                else:
                    assert p == q, f"{c.name}: cell {i} differs between the specialised and the generic path"
