"""Stats sums at the limit of the exact integer path.

A stats cell over an integer column of at most QW_SUM_EXACT_BITS bits used to add the raw offsets in a
uint64. A multi-valued column sums values, not docs, so an ordinary split can hold enough values for that
sum to wrap, and the finished `sum` / `avg` came out as the exact sum mod 2^64. The oracle and the kernels
wrapped the same way, so GPU == oracle could not see it. This test compares the finished aggregation with
an exact Python-int sum of the values the test generated."""
import numpy as np

from quickwit_b200 import ffi, splitgen as S
from pipeline import MATCH_ALL, cpu_root_search

MAPPING = {"field_mappings": [{"name": "v", "type": "u64", "fast": True}]}


def _multi_40bit_split(num_docs=3_000_000, per_doc=6, seed=7):
    """num_docs * per_doc values of a 40-bit raw span (one value is 0, the others near 2^40): the exact sum
    of the raws is about 1.07 * 2^64."""
    rng = np.random.default_rng(seed)
    vals = (1 << 40) - 1 - rng.integers(0, 1 << 20, size=num_docs * per_doc, dtype=np.uint64)
    vals[0] = 0
    start = np.arange(0, num_docs * per_doc + 1, per_doc, dtype=np.uint32)
    b = S._Builder(num_docs)
    b.add_column("v", ffi.COL_U64, ffi.CARD_MULTI, vals, start)
    return b.finish("multi-40"), vals


def _exact_sum(vals: np.ndarray) -> int:
    # split each value into 20-bit halves so that the numpy sums stay far below 2^64
    lo = int((vals & np.uint64((1 << 20) - 1)).sum(dtype=np.uint64))
    hi = int((vals >> np.uint64(20)).sum(dtype=np.uint64))
    return (hi << 20) + lo


def test_multivalued_40_bit_sum_beyond_2_64():
    img, vals = _multi_40bit_split()
    col = img.columns()[img.column_ord("v")]
    assert col.bits == 40 and col.num_vals == len(vals) and col.cardinality == ffi.CARD_MULTI
    exact = _exact_sum(vals)
    assert exact >= 1 << 64, "the case must overflow a uint64 sum of raws"
    aggs = {"s": {"stats": {"field": "v"}}, "a": {"avg": {"field": "v"}}, "t": {"sum": {"field": "v"}}}
    out = cpu_root_search([img], MATCH_ALL, MAPPING, max_hits=0, aggs=aggs)["aggregations"]
    n = len(vals)
    bound = n * 2.0 ** -52 * exact  # f64 accumulation in value order
    st = out["s"]
    assert st["count"] == n
    assert st["min"] == 0.0 and st["max"] == float(int(vals.max()))
    assert abs(st["sum"] - exact) <= bound, f"sum {st['sum']!r} vs exact {exact} (wrapped: {exact % (1 << 64)})"
    assert abs(out["t"]["value"] - exact) <= bound
    assert abs(st["avg"] - exact / n) <= bound / n
    assert abs(out["a"]["value"] - exact / n) <= bound / n
