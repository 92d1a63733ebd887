"""C-ABI surface + host-only logic (no GPU): every symbol declared in include/qwgpu.h is exported,
the product fails loudly without a device, and the independent Python / C++ protobuf codecs and
the query compiler agree."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

from quickwit_b200 import ffi, plan as P, proto, service, splitgen as S
from quickwit_b200.proto import ASC, DESC
from oracle import oracle as O
from pipeline import MATCH_ALL, bool_, full_text, search_request, term

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_declared_symbol_is_exported():
    hdr = open(os.path.join(ROOT, "include", "qwgpu.h")).read()
    names = sorted(set(re.findall(r"\b(qwgpu_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 25
    L = C.CDLL(ffi.LIB_PATH)
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_no_cpu_fallback():
    import torch
    if torch.cuda.device_count() > 0:  # (asked of the CUDA runtime: a GPU's device node need not be /dev/nvidia0)
        pytest.skip("a GPU is present")
    with pytest.raises(ffi.QwGpuError) as e:
        service.SearcherContext(0)
    assert e.value.code == ffi.ENODEVICE
    ctx = service.SearcherContext(None)  # host-only context
    img = S.synth_split(2000, 0, [0.1])
    with pytest.raises(ffi.QwGpuError) as e:
        ctx.register_split(img)
    assert e.value.code == ffi.ENODEVICE
    with pytest.raises(ffi.QwGpuError) as e:
        ctx.leaf_search(proto.enc_leaf_search_request(search_request(MATCH_ALL, max_hits=1), [], "{}"))
    assert e.value.code == ffi.ENODEVICE


def test_product_does_not_reference_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "quickwit_b200")):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".h")) or f == "Makefile":
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "qworacle" not in text and "from oracle" not in text and "import oracle" not in text, f


def test_compiled_plan_matches_hand_built_plan():
    img = S.synth_split(5000, 3, [0.2, 0.1, 0.05], split_id="cp")
    dm = json.dumps({"field_mappings": [], "timestamp_field": "timestamp"})
    ast = bool_(should=[term("body", "t0"), term("body", "t1"), term("body", "t2")])
    got = service.compile_plan(img, search_request(ast, max_hits=10, sort_fields=[("_score", DESC)]), dm)
    root = P.bool_([P.term(img, "body", f"t{i}", occur=ffi.OCCUR_SHOULD) for i in range(3)])
    want = P.make_plan(root, 10, [(ffi.SORT_SCORE, ffi.ORDER_DESC, ffi.ABSENT)])
    assert got == want
    # same results through the oracle, including the f32 BM25 weights computed by the C++ host
    a, b = O.split_search(img, got), O.split_search(img, want)
    assert a.hits == b.hits and a.num_hits == b.num_hits


def test_bool_simplification_rules():
    """TantivyBoolQuery::simplify (tantivy_query_ast.rs:190-337), observed through compiled plans."""
    img = S.synth_split(3000, 1, [0.3, 0.2], split_id="simp")
    dm = "{}"
    node = lambda pl, i: ffi.QwPlanNode.from_buffer_copy(pl[C.sizeof(ffi.QwPlanHeader) + i * C.sizeof(ffi.QwPlanNode):][:C.sizeof(ffi.QwPlanNode)])
    nn = lambda pl: ffi.QwPlanHeader.from_buffer_copy(pl[:C.sizeof(ffi.QwPlanHeader)]).num_nodes
    comp = lambda ast, **kw: service.compile_plan(img, search_request(ast, max_hits=1, **kw), dm)
    assert node(comp(bool_()), 0).kind == ffi.NODE_ALL                         # empty bool == match_all
    assert node(comp(bool_(must=[{"type": "match_none"}, term("body", "t0")])), 0).kind == ffi.NODE_NONE
    pl = comp(bool_(must=[term("body", "t0")]))                                 # single must clause is unwrapped
    assert nn(pl) == 1 and node(pl, 0).kind == ffi.NODE_TERM
    pl = comp(bool_(filter=[term("body", "t0")]))                               # a single filter is NOT unwrapped (keeps score 0)
    assert node(pl, 0).kind == ffi.NODE_BOOL and node(pl, 1).occur == ffi.OCCUR_FILTER
    pl = comp(bool_(must=[bool_(must=[term("body", "t0")], must_not=[term("body", "t1")])]))  # nested must flattened
    assert node(pl, 0).kind == ffi.NODE_BOOL and node(pl, 0).num_children == 2
    pl = comp(bool_(must_not=[term("body", "t0")]))                             # only must_not: match_all is added
    kinds = sorted(node(pl, i).kind for i in range(1, nn(pl)))
    assert node(pl, 0).kind == ffi.NODE_BOOL and kinds == [ffi.NODE_TERM, ffi.NODE_ALL]
    assert node(comp(bool_(should=[], minimum_should_match=1)), 0).kind == ffi.NODE_NONE
    dm_ts = json.dumps({"timestamp_field": "timestamp", "field_mappings": [{"name": "timestamp", "type": "datetime", "fast": True}]})
    pl = service.compile_plan(img, search_request(term("body", "t0"), max_hits=1, start_timestamp=1_700_000_010, end_timestamp=1_700_000_020), dm_ts)
    assert node(pl, 0).kind == ffi.NODE_BOOL and node(pl, 2).kind == ffi.NODE_RANGE and node(pl, 2).occur == ffi.OCCUR_FILTER
    assert (S.u64_to_i64(node(pl, 2).lo), S.u64_to_i64(node(pl, 2).hi)) == (1_700_000_010 * 10**9, 1_700_000_020 * 10**9 - 1)
    with pytest.raises(ffi.QwGpuError) as e:
        comp({"type": "bool", "must": [{"type": "nope"}]})
    assert e.value.code == ffi.EINVALID_QUERY


def test_python_and_cpp_protobuf_codecs_agree():
    hits = [{"split_id": "s1", "segment_ord": 0, "doc_id": 7, "sort_value": ("f64", 1.5), "sort_value2": ("i64", -3)},
            {"split_id": "s0", "segment_ord": 0, "doc_id": 9, "sort_value": ("u64", 2**63 + 5)},
            {"split_id": "s2", "segment_ord": 0, "doc_id": 1, "sort_value": None, "sort_value2": ("bool", True)}]
    resp = proto.enc_leaf_search_response(42, hits, [("boom", "s9", True)], 3, 2, b"\x00\x01agg")
    req = proto.enc_search_request("{}", max_hits=10, sort_fields=[("a", DESC), ("b", ASC)])
    # single-response shortcut: decoded by the C++ codec, re-encoded, decoded by the Python codec
    out = proto.dec_leaf_search_response(service.merge_leaf_responses(req, [resp]))
    assert out["num_hits"] == 42 and out["partial_hits"] == hits and out["intermediate_aggregation_result"] == b"\x00\x01agg"
    assert out["failed_splits"] == [{"error": "boom", "split_id": "s9", "retryable_error": True}]
    assert (out["num_attempted_splits"], out["num_successful_splits"]) == (3, 2)


def test_heterogeneous_sort_value_order():
    """SortValue::cmp across types (quickwit-proto/src/search/mod.rs:137-161; root.rs:3329-3692)."""
    mk = lambda i, sv: {"split_id": "s", "segment_ord": 0, "doc_id": i, "sort_value": sv}
    vals = [("u64", 2**63 + 1), ("i64", -5), ("f64", 2.5), ("u64", 3), ("i64", 2), ("bool", True), ("f64", -7.25), None]
    parts = [proto.enc_leaf_search_response(1, [mk(i, v)], num_attempted_splits=1, num_successful_splits=1) for i, v in enumerate(vals)]
    req = lambda o: proto.enc_search_request("{}", max_hits=8, sort_fields=[("f", o)])
    order = lambda o: [h["doc_id"] for h in proto.dec_leaf_search_response(service.merge_leaf_responses(req(o), parts))["partial_hits"]]
    assert order(DESC) == [0, 3, 2, 4, 5, 1, 6, 7]   # 2^63+1 > 3 > 2.5 > 2 > true(1) > -5 > -7.25 > None
    assert order(ASC) == [6, 1, 5, 4, 2, 3, 0, 7]    # None stays last in both directions


def test_posting_and_column_format_roundtrip():
    rng = np.random.default_rng(3)
    n = 70_000
    b = S._Builder(n)
    fid = b.add_field("f", ffi.FIELD_HAS_FREQS, ffi.TOK_RAW, None, n)
    lists = {}
    for name, p in (("dense", 0.7), ("mid", 0.03), ("rare", 0.0002), ("all", 1.0), ("one", None)):
        docs = np.array([n - 1], dtype=np.uint32) if p is None else np.nonzero(rng.random(n) < p)[0].astype(np.uint32)
        tfs = rng.integers(1, 2000, size=len(docs)).astype(np.uint32)
        lists[name] = (docs, tfs)
        b.add_term(fid, name.encode(), docs, tfs)
    vals = rng.integers(0, 2**40, size=n).astype(np.uint64) * 3 + 11
    b.add_column("full", ffi.COL_U64, ffi.CARD_FULL, vals, None)
    some = np.nonzero(rng.random(n) < 0.3)[0].astype(np.uint32)
    b.add_column("opt", ffi.COL_I64, ffi.CARD_OPTIONAL, np.array([S.i64_to_u64(int(x) - 50) for x in some], dtype=np.uint64), some)
    wide = rng.integers(0, 2**63, size=n).astype(np.uint64) * 2 + rng.integers(0, 2, size=n).astype(np.uint64)
    wide[0], wide[1] = 0, 2**64 - 1
    b.add_column("wide", ffi.COL_U64, ffi.CARD_FULL, wide, None)
    img = b.finish("fmt")
    for name, (docs, tfs) in lists.items():
        d, t = O.decode_postings(img, img.term_ord("f", name), n)
        assert np.array_equal(d, docs) and np.array_equal(t, tfs), name
    v, p = O.column_first(img, img.column_ord("full"))
    assert p.all() and np.array_equal(v, vals)
    c = img.columns()[img.column_ord("full")]
    assert c.gcd == 3 and c.min_value == vals.min()
    v, p = O.column_first(img, img.column_ord("opt"))
    assert np.array_equal(np.nonzero(p)[0], some) and [S.u64_to_i64(int(x)) for x in v[p][:5]] == [int(x) - 50 for x in some[:5]]
    assert img.columns()[img.column_ord("wide")].bits == 64
    v, p = O.column_first(img, img.column_ord("wide"))
    assert np.array_equal(v, wide)


def test_partial_hit_wire_form_every_value_kind_and_long_split_ids():
    """The C encoder of LeafSearchResponse.partial_hits against the pure-Python codec: every SortByValue
    kind incl. 10-byte varints, absent sort values, and split ids longer than the encoder's stack buffer."""
    from quickwit_b200 import proto, service
    hits = []
    for i, sid in enumerate(["s", "01HZXJ5QK8W9D3M7P2R4T6V8YB", "x" * 150, "y" * 400]):
        hits += [
            {"split_id": sid, "segment_ord": 0, "doc_id": i, "sort_value": ("u64", 2**64 - 1 - i), "sort_value2": ("i64", -(2**63) + i)},
            {"split_id": sid, "segment_ord": 0, "doc_id": 100 + i, "sort_value": ("f64", -1.5e300 * (i + 1)), "sort_value2": ("bool", True)},
            {"split_id": sid, "segment_ord": 0, "doc_id": 0},
        ]
    req = proto.enc_search_request('{"type": "match_all"}', max_hits=100)
    resp = proto.enc_leaf_search_response(num_hits=len(hits), partial_hits=hits, num_attempted_splits=1, num_successful_splits=1)
    out = proto.dec_leaf_search_response(service.merge_leaf_responses(req, [resp]))   # single-response shortcut: order kept
    got = [{k: v for k, v in h.items() if v is not None} for h in out["partial_hits"]]
    want = [{k: v for k, v in h.items()} for h in hits]
    assert got == want


def test_corrupt_split_images_are_rejected():
    """Every offset of a split image is checked before it is followed (they end up as device pointers):
    truncated images and out-of-range sections / terms / columns fail with EINVALID_ARG."""
    img = S.synth_split(5000, 3, [0.2, 0.1], split_id="corrupt")
    dm = json.dumps({"field_mappings": [], "timestamp_field": "timestamp"})
    req = search_request(term("body", "t0"), max_hits=3)
    assert service.compile_plan(img, req, dm)
    hdr = img.header()
    H, T, CO = ffi.QwImgHeader, ffi.QwImgTerm, ffi.QwImgColumn

    def broken(mutate):
        raw = img.array.copy()
        mutate(raw)
        with pytest.raises(ffi.QwGpuError) as e:
            service.compile_plan(S.SplitImage(raw, "corrupt"), req, dm)
        assert e.value.code == ffi.EINVALID_ARG, e.value.msg

    def put64(raw, off, v):
        raw[off:off + 8] = np.frombuffer(np.uint64(v).tobytes(), dtype=np.uint8)

    with pytest.raises(ffi.QwGpuError):
        service.compile_plan(S.SplitImage(img.array[: img.nbytes - 64].copy(), "corrupt"), req, dm)
    broken(lambda r: put64(r, H.terms_off.offset, hdr.total_len - 8))
    broken(lambda r: put64(r, H.data_len.offset, hdr.data_len + 4096))
    broken(lambda r: put64(r, H.strings_len.offset, 1 << 40))
    broken(lambda r: put64(r, hdr.terms_off + T.data_off.offset, hdr.data_len))            # first term: blocks past the data region
    broken(lambda r: put64(r, hdr.terms_off + T.widx_off.offset, hdr.data_len - 8))
    broken(lambda r: put64(r, hdr.columns_off + CO.values_off.offset, hdr.data_len - 8))
    broken(lambda r: put64(r, hdr.columns_off + CO.index_len.offset, 1 << 50))


def test_unsupported_requests_are_not_marked_retryable():
    """leaf.rs:1989-2004 marks failed splits retryable so that the root re-runs them on another node; a
    request this library does not execute would fail there the same way (the C++ side reports it with
    retryable_error = false). Checked on the source: the leaf path needs a device."""
    src = open(os.path.join(ROOT, "quickwit_b200", "csrc", "leaf.cpp")).read()
    assert "return code != QWGPU_EUNSUPPORTED" in src
    assert not re.search(r"failed\.push_back\(\{[^}]*, true\}\)", src)


def _optimized(ast, splits, mapping=None, **req_kw):
    """splits: [(split_id, num_docs, ts_start, ts_end)] -> qwgpu_optimize_leaf_request rows"""
    mapping = mapping or {"field_mappings": [{"name": "ts", "type": "datetime", "fast": True}, {"name": "body", "type": "text"},
                                             {"name": "n", "type": "u64", "fast": True}], "timestamp_field": "ts"}
    offsets = [proto.enc_split_offsets(sid, nd, a, b) for sid, nd, a, b in splits]
    return service.optimize_leaf_request(proto.enc_leaf_search_request(search_request(ast, **req_kw), offsets, json.dumps(mapping)))


def test_can_split_do_better_static_pruning():
    """CanSplitDoBetter::optimize (leaf.rs:1141-1242) + is_metadata_count_request_with_ast (root.rs:665-686)."""
    row = lambda r: (r["split_id"], r["hits_disabled"], r["metadata_count"])
    # no sort: splits in descending split-id order; once the doc counts reach start_offset + max_hits the rest only count
    got = _optimized(MATCH_ALL, [("a", 2, None, None), ("b", 5, None, None), ("c", 1, None, None), ("0", 9, None, None)], max_hits=2, start_offset=1)
    assert [row(r) for r in got] == [("c", False, False), ("b", False, False), ("a", True, True), ("0", True, True)]
    assert [r["max_hits"] for r in got] == [2, 2, 0, 0]
    # the first split alone is enough
    got = _optimized(MATCH_ALL, [("a", 2, None, None), ("b", 5, None, None)], max_hits=5)
    assert [row(r) for r in got] == [("b", False, False), ("a", True, True)]
    # sort by the timestamp field, descending: order by timestamp_end desc; a later split is demoted only when it
    # ends before every required split starts (ranges may overlap)
    splits = [("s1", 5, 0, 4), ("s2", 5, 11, 20), ("s3", 5, 5, 25), ("s4", 5, 3, 9)]
    got = _optimized(MATCH_ALL, splits, max_hits=4, sort_fields=[("ts", DESC)])
    assert [row(r) for r in got] == [("s3", False, False), ("s2", False, False), ("s4", False, False), ("s1", True, True)]
    got = _optimized(MATCH_ALL, splits, max_hits=7, sort_fields=[("ts", DESC)])   # two splits required: smallest start = 5
    assert [row(r) for r in got] == [("s3", False, False), ("s2", False, False), ("s4", False, False), ("s1", True, True)]
    # ascending: order by timestamp_start; demoted when it starts after every required split has ended
    got = _optimized(MATCH_ALL, splits, max_hits=4, sort_fields=[("ts", ASC)])
    assert [row(r) for r in got] == [("s1", False, False), ("s4", False, False), ("s3", True, True), ("s2", True, True)]
    got = _optimized(MATCH_ALL, splits, max_hits=6, sort_fields=[("ts", ASC)])    # s1 + s4 required: biggest end = 9
    assert [row(r) for r in got] == [("s1", False, False), ("s4", False, False), ("s3", False, False), ("s2", True, True)]
    # a sort field that is not the timestamp field says nothing: request order, nothing demoted
    got = _optimized(MATCH_ALL, splits, max_hits=1, sort_fields=[("n", DESC)])
    assert [row(r) for r in got] == [(s[0], False, False) for s in splits]
    # not a match-all query / time bounds / aggregation / search_after: ordered, never demoted
    got = _optimized(term("body", "x"), splits, max_hits=1, sort_fields=[("ts", DESC)])
    assert [row(r) for r in got] == [("s3", False, False), ("s2", False, False), ("s4", False, False), ("s1", False, False)]
    for kw in (dict(start_timestamp=3), dict(end_timestamp=30), dict(aggs={"c": {"terms": {"field": "n"}}}),
               dict(search_after={"split_id": "s2", "segment_ord": 0, "doc_id": 1, "sort_value": ("i64", 5)})):
        got = _optimized(MATCH_ALL, splits, max_hits=1, sort_fields=[("ts", DESC)], **kw)
        assert not any(r["hits_disabled"] or r["metadata_count"] for r in got), kw
    # count requests: match-all without bounds or aggregations is answered from num_docs
    assert all(r["metadata_count"] for r in _optimized(MATCH_ALL, splits, max_hits=0))
    assert not any(r["metadata_count"] for r in _optimized(MATCH_ALL, splits, max_hits=0, aggs={"c": {"terms": {"field": "n"}}}))
    assert not any(r["metadata_count"] for r in _optimized(MATCH_ALL, splits, max_hits=0, end_timestamp=7))
    assert not any(r["metadata_count"] for r in _optimized(term("body", "x"), splits, max_hits=0))


def test_underestimate_count_skips_splits_with_nothing_left_to_compute():
    """simplify_search_request (leaf.rs:1399-1433): under CountHits::Underestimate a split whose hits were disabled (or
    never wanted) and that has no aggregation to feed is pruned before warmup; CountAll keeps it as a count request."""
    UNDER = 1
    splits = [("a", 2, None, None), ("b", 5, None, None), ("c", 1, None, None), ("0", 9, None, None)]
    row = lambda r: (r["split_id"], r["hits_disabled"], r["metadata_count"], r["skipped"])
    got = _optimized(MATCH_ALL, splits, max_hits=2, start_offset=1, count_hits=UNDER)
    assert [row(r) for r in got] == [("c", False, False, False), ("b", False, False, False), ("a", True, False, True), ("0", True, False, True)]
    got = _optimized(MATCH_ALL, splits, max_hits=2, start_offset=1)   # CountAll: counted from the metadata instead
    assert [row(r) for r in got] == [("c", False, False, False), ("b", False, False, False), ("a", True, True, False), ("0", True, True, False)]
    # an aggregation keeps every split; a term query is never demoted, so nothing is skipped while hits are wanted
    assert not any(r["skipped"] for r in _optimized(MATCH_ALL, splits, max_hits=2, count_hits=UNDER, aggs={"c": {"terms": {"field": "n"}}}))
    assert not any(r["skipped"] for r in _optimized(term("body", "x"), splits, max_hits=2, count_hits=UNDER))
    # a pure count request under Underestimate computes nothing at all (the reference returns Some only for CountAll)
    assert all(r["skipped"] for r in _optimized(term("body", "x"), splits, max_hits=0, count_hits=UNDER))
    assert not any(r["skipped"] for r in _optimized(term("body", "x"), splits, max_hits=0))


def test_partial_exchange_carries_failed_splits_and_rejects_corrupt_partials():
    """The fixed-size per-rank partial (SURVEY.md 8e): hits, aggregation bytes, failed_splits entries and resource
    statistics survive response -> partial -> merge; sizes claimed inside a gathered partial are checked."""
    import torch
    hit = lambda split, doc, v: {"split_id": split, "segment_ord": 0, "doc_id": doc, "sort_value": ("i64", v)}
    req = search_request(MATCH_ALL, max_hits=3, sort_fields=[("ts", DESC)])
    stats = lambda cpu: proto.enc_leaf_resource_stats(cpu, cpu, 1)
    r0 = proto.enc_leaf_search_response(10, [hit("a", 1, 50), hit("a", 2, 40)], [("boom", "x-1", True), ("nope", "x-2", False)], 4, 2, resource_stats=stats(100))
    r1 = proto.enc_leaf_search_response(7, [hit("b", 9, 45)], [], 1, 1, resource_stats=stats(30))
    nbytes = service.partial_size(req)
    buf = torch.zeros(2 * nbytes, dtype=torch.uint8)
    service.response_to_partial(req, r0, buf.data_ptr(), nbytes)
    service.response_to_partial(req, r1, buf.data_ptr() + nbytes, nbytes)
    out = proto.dec_leaf_search_response(service.merge_partials(req, 2, buf.data_ptr(), nbytes))
    want = proto.dec_leaf_search_response(service.merge_leaf_responses(req, [r0, r1]))
    assert out == want
    assert out["failed_splits"] == [{"error": "boom", "split_id": "x-1", "retryable_error": True}, {"error": "nope", "split_id": "x-2", "retryable_error": False}]
    assert (out["num_attempted_splits"], out["num_successful_splits"]) == (5, 3)
    assert out["resource_stats"]["split_resources_sum"]["cpu_search_microsecs"] == 130
    # corrupt counts inside a gathered partial: n_hits > k, aggregation length, tail length, failed-split count
    for word, value in ((8, 4), (9, 1 << 24), (11, 1 << 20), (10, 7)):
        bad = buf.clone()
        bad.view(torch.int32)[word] = value
        with pytest.raises(ffi.QwGpuError) as e:
            service.merge_partials(req, 2, bad.data_ptr(), nbytes)
        assert e.value.code == ffi.EINVALID_ARG, (word, e.value.msg)
    # more failed splits than the tail holds: refused at the sender, never truncated
    many = proto.enc_leaf_search_response(0, [], [("e" * 60, f"split-{i:04d}", True) for i in range(100)], 100, 0)
    with pytest.raises(ffi.QwGpuError) as e:
        service.response_to_partial(req, many, buf.data_ptr(), nbytes)
    assert e.value.code == ffi.EUNSUPPORTED


def test_split_bundle_footer():
    """A `.split` file's footer built byte by byte the way the reference writes it (bundle_storage.rs:92-174:
    versioned header magic 403881646 / version 1 + JSON, u32 length; hot_directory.rs:40-80: magic 2557869106 /
    version 1, u32 length, postcard HotDirectoryMeta, slices; u32 length) and read back."""
    import struct
    files = {"a.term": b"T" * 100, "a.idx": b"I" * 3000, "a.pos": b"P" * 70, "b.fast": b"F" * 555, "meta.json": b"{}"}
    body, ranges = b"", {}
    for name, data in files.items():
        ranges[name] = {"start": len(body), "end": len(body) + len(data)}
        body += data
    meta = struct.pack("<II", 403881646, 1) + json.dumps({"files": ranges}).encode()

    def varint(v):
        out = b""
        while True:
            b7 = v & 0x7F
            v >>= 7
            out += bytes([b7 | (0x80 if v else 0)])
            if not v:
                return out
    pstr = lambda s: varint(len(s)) + s.encode()
    file_lengths = {"a.term": 100, "a.idx": 3000, "b.fast": 555}
    slice_offsets = [("a.term", 0), ("a.idx", 130), ("b.fast", 400)]
    pc = varint(len(file_lengths)) + b"".join(pstr(k) + varint(v) for k, v in file_lengths.items())
    pc += varint(len(slice_offsets)) + b"".join(pstr(k) + varint(v) for k, v in slice_offsets)
    slices = b"S" * 1000
    hot = struct.pack("<III", 2557869106, 1, len(pc)) + pc + slices
    split = body + meta + struct.pack("<I", len(meta)) + hot + struct.pack("<I", len(hot))
    footer_start = len(body)
    for tail_from in (footer_start, 0, footer_start - 17):      # exactly the footer, the whole file, a bit more than the footer
        got = service.parse_split_footer(split[tail_from:], len(split))
        assert [(f["path"], f["start"], f["end"]) for f in got["files"]] == [(k, v["start"], v["end"]) for k, v in ranges.items()]
        assert got["footer_start"] == footer_start and got["footer_end"] == len(split)
        assert got["bundle_metadata"] == {"offset": footer_start, "len": len(meta)}
        h = got["hotcache"]
        assert h["offset"] == footer_start + len(meta) + 4 and h["len"] == len(hot) and h["file_lengths"] == file_lengths
        first_slice = h["offset"] + 12 + len(pc)
        assert [(s["path"], s["offset"]) for s in h["slices"]] == [(k, first_slice + o) for k, o in slice_offsets]
        assert split[h["slices"][0]["offset"]:h["slices"][0]["offset"] + 4] == b"SSSS"
    # corrupt footers are rejected, not followed
    bad = bytearray(split)
    bad[footer_start] ^= 0xFF                                    # bundle magic
    with pytest.raises(ffi.QwGpuError) as e:
        service.parse_split_footer(bytes(bad[footer_start:]), len(split))
    assert e.value.code == ffi.EINVALID_ARG and "magic number" in e.value.msg
    for cut in (3, 40, len(split) - footer_start - 10):         # the tail does not hold the whole footer
        with pytest.raises(ffi.QwGpuError):
            service.parse_split_footer(split[-cut:], len(split))
    bad = bytearray(split)
    bad[-4:] = struct.pack("<I", len(split) + 5)                 # hotcache longer than the file
    with pytest.raises(ffi.QwGpuError):
        service.parse_split_footer(bytes(bad[footer_start:]), len(split))


def test_synthetic_positions_field_is_deterministic_and_consistent():
    """qwgpu_synth_split with msg_vocab > 0 (the positions field behind BASELINE config 5's phrase queries): same
    spec => same bytes; without it the image is the plain corpus; a phrase can only match
    documents that hold all of its words."""
    from quickwit_b200 import plan as P
    from oracle import oracle as O
    a = S.synth_split(30_000, 3, [0.2, 0.05], split_id="m", msg_vocab=32)
    b = S.synth_split(30_000, 3, [0.2, 0.05], split_id="m", msg_vocab=32)
    plain = S.synth_split(30_000, 3, [0.2, 0.05], split_id="m")
    assert a.array.tobytes() == b.array.tobytes() and plain.nbytes < a.nbytes
    by_doc = [(ffi.SORT_DOCID, ffi.ORDER_DESC, ffi.ABSENT)]
    n = lambda root, img=a: O.split_search(img, P.make_plan(root, 0, by_doc)).num_hits
    assert 0 < n(P.phrase(a, "msg", ["w3", "w3"])) < n(P.term(a, "msg", "w3"))   # the word twice in a row: a subset
    both = n(P.bool_([P.term(a, "msg", "w1", occur=ffi.OCCUR_MUST), P.term(a, "msg", "w2", occur=ffi.OCCUR_MUST)]))
    ph12, ph21 = n(P.phrase(a, "msg", ["w1", "w2"])), n(P.phrase(a, "msg", ["w2", "w1"]))
    assert 0 < ph12 <= both and 0 < ph21 <= both
    # the body terms are untouched by the extra field
    assert n(P.term(a, "body", "t0")) == n(P.term(plain, "body", "t0"), plain)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): exactly one JSON line on stdout
    with the contract's keys and the same workload description as the GPU arm."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--splits", "2", "--docs-per-split", "50000"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "docs_scored_per_sec" and d["unit"] == "postings/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 2 and d["config"]["workload"] == "c2_bm25_or10_top1000"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "postings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_refuses_arguments_it_cannot_honour():
    """--steps below 1 would time nothing; --dump-outputs writes the outputs of the GPU arm only."""
    import subprocess
    import sys
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr, extra


def test_bench_dump_sample_is_seeded_and_within_budget(tmp_path):
    """Outputs larger than --dump-outputs' 64 MB are written as a fixed sample of their rows, in order."""
    import bench
    big = np.arange(12_000_000, dtype=np.float64).reshape(-1, 4)      # 96 MB
    small = np.arange(8, dtype=np.float64)
    bench.write_outputs(str(tmp_path / "a"), {"big": big, "small": small})
    bench.write_outputs(str(tmp_path / "b"), {"big": big, "small": small})
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert np.array_equal(a, b) and len(a) < len(big) and np.all(np.diff(a[:, 0]) > 0) and np.all(a[:, 0] % 4 == 0)
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small)


def test_wildcard_queries_expand_over_the_split_dictionary():
    """WildcardQuery (quickwit-query/src/query_ast/wildcard_query.rs): `*` / `?` / backslash escapes, text parts through the
    field tokenizer's normalizer (default: lower-cased, raw: unchanged), case_insensitive, lenient; matching documents
    compared with a brute force over the documents' tokens. Constant-score semantics: refused under BM25 ranking in a
    scoring position (like term_set), fine as a filter or under any other sort."""
    mapping = {"field_mappings": [{"name": "body", "type": "text", "record": "freq", "fieldnorms": True},
                                  {"name": "tag", "type": "text", "tokenizer": "raw"}, {"name": "n", "type": "u64", "fast": True}]}
    words = ["alpha", "alpine", "beta", "betamax", "gamma", "Alphabet", "al", "élan", "a*b", "delta"]
    tags = ["Prod-EU", "prod-us", "Dev", "staging?"]
    docs = [{"body": f"{words[i % 10]} {words[(i * 3) % 10]} filler", "tag": tags[i % 4], "n": i} for i in range(200)]
    img = S.build_split(docs, mapping, "wc-0")
    dm = json.dumps(mapping)

    def run(ast, **kw):
        return O.split_search(img, service.compile_plan(img, search_request(ast, **kw), dm))

    def to_regex(pat):  # the reference's translation: text escaped, `*` -> `.*`, `?` -> `.`
        out, i = "", 0
        while i < len(pat):
            c = pat[i]
            if c == "*":
                out += ".*"
            elif c == "?":
                out += "."
            elif c == "\\":
                if i + 1 >= len(pat):
                    break
                out += re.escape(pat[i + 1]); i += 1
            else:
                out += re.escape(c)
            i += 1
        return out

    def brute(field, pat, ci=False):
        if field == "body":
            rx = re.compile(to_regex(pat.lower() if not ci else pat.lower()), re.S)
            toks = lambda d: [t.lower() for t in re.findall(r"[^\W_]+", d["body"], re.U)]
        else:
            rx = re.compile(to_regex(pat), re.S | (re.I if ci else 0))
            toks = lambda d: [d["tag"]]
        return sorted((i for i, d in enumerate(docs) if any(rx.fullmatch(t) for t in toks(d))), reverse=True)

    wc = lambda field, value, **kw: {"type": "wildcard", "field": field, "value": value, **kw}
    for field, pat, ci in [("body", "al*", False), ("body", "AL*", False), ("body", "?eta", False), ("body", "*ma*", False), ("body", "a\\*b", False),
                           ("body", "é?an", False), ("body", "*", False), ("body", "zz*", False), ("tag", "prod*", False), ("tag", "Prod*", False),
                           ("tag", "prod*", True), ("tag", "staging\\?", False), ("tag", "stag*\\", False), ("tag", "???", False)]:
        r = run(wc(field, pat, case_insensitive=ci), max_hits=200)
        want = brute(field, pat, ci)
        assert r.num_hits == len(want) and [h[0] for h in r.hits] == want, (field, pat, ci, r.num_hits, len(want))
    assert run(wc("body", "al*"), max_hits=0).num_hits == 120
    # scoring: refused in a scoring position under BM25 ranking, accepted as a filter
    with pytest.raises(ffi.QwGpuError) as ei:
        run(wc("body", "al*"), max_hits=5, sort_fields=[("_score", DESC)])
    assert ei.value.code == ffi.EUNSUPPORTED
    with pytest.raises(ffi.QwGpuError):
        run({"type": "term_set", "terms_per_field": {"body": ["alpha", "beta"]}}, max_hits=5, sort_fields=[("_score", DESC)])
    flt = run(bool_(must=[term("body", "filler")], filter=[wc("body", "al*")]), max_hits=5, sort_fields=[("_score", DESC)])
    assert flt.num_hits == 120
    assert run({"type": "term_set", "terms_per_field": {"body": ["alpha", "beta"]}}, max_hits=0).num_hits == len(brute("body", "alpha", False) + [i for i in brute("body", "beta", False) if i not in brute("body", "alpha", False)])
    # the reference's own translation vectors (wildcard_query.rs:224-302: "MyString Wh1ch?a.nOrMal Tokenizer would*cut" ->
    # `MyString Wh1ch.a\.nOrMal Tokenizer would.*cut` on a raw field, everything escaped when `?` / `*` are escaped),
    # checked as behaviour on raw terms: `.` stays a literal, `?` is one character, `*` any run
    vec_docs = [{"tag": t, "body": "x", "n": i} for i, t in enumerate([
        "MyString Wh1chXa.nOrMal Tokenizer wouldZZcut", "MyString Wh1ch?a.nOrMal Tokenizer would*cut",
        "MyString Wh1chXaXnOrMal Tokenizer wouldcut", "mystring wh1chxa.normal tokenizer wouldcut", "MyString Wh1cha.nOrMal Tokenizer wouldcut"])]
    vimg = S.build_split(vec_docs, mapping, "wc-vec")
    vrun = lambda value: sorted(h[0] for h in O.split_search(vimg, service.compile_plan(vimg, search_request(wc("tag", value), max_hits=10), dm)).hits)
    assert vrun("MyString Wh1ch?a.nOrMal Tokenizer would*cut") == [0, 1]
    assert vrun("MyString Wh1ch\\?a.nOrMal Tokenizer would\\*cut") == [1]
    # errors and leniency
    with pytest.raises(ffi.QwGpuError) as ei:
        run(wc("n", "1*"), max_hits=0)
    assert ei.value.code == ffi.EINVALID_QUERY and "non-text" in ei.value.msg
    with pytest.raises(ffi.QwGpuError):
        run(wc("nope", "x*"), max_hits=0)
    assert run(wc("nope", "x*", lenient=True), max_hits=0).num_hits == 0


def test_merge_leaf_responses_against_an_independent_restatement_of_the_order():
    """Root / leaf merge at scale (collector.rs:914-992, 1120-1153; SortOrder::compare_opt, quickwit-proto/src/lib.rs:122-140):
    random per-leaf hit lists with ties, None sort values, one or two sort keys and both directions — qwgpu_merge_leaf_responses
    against a Python restatement written from the reference's comparator, not from the product's code."""
    import functools
    import random
    rng = random.Random(7)

    def cmp_opt(a, b, order):  # greater = better; Some beats None in both directions
        if a is None or b is None:
            return (a is not None) - (b is not None)
        return ((a > b) - (a < b)) * (1 if order == DESC else -1)

    def better(x, y, o1, o2):
        c = cmp_opt(x.get("sort_value", (None, None))[1] if x.get("sort_value") else None,
                    y.get("sort_value", (None, None))[1] if y.get("sort_value") else None, o1)
        if c == 0:
            c = cmp_opt(x.get("sort_value2", (None, None))[1] if x.get("sort_value2") else None,
                        y.get("sort_value2", (None, None))[1] if y.get("sort_value2") else None, o2)
        if c == 0:
            ax, ay = (x["split_id"], x["segment_ord"], x["doc_id"]), (y["split_id"], y["segment_ord"], y["doc_id"])
            c = ((ax > ay) - (ax < ay)) * (1 if o1 == DESC else -1)
        return c

    for trial in range(60):
        o1, o2 = rng.choice([ASC, DESC]), rng.choice([ASC, DESC])
        two = rng.random() < 0.5
        k = rng.choice([1, 3, 10, 40])
        leaves, everything, total = [], [], 0
        for leaf in range(rng.randint(1, 6)):
            hits = []
            for _ in range(rng.randint(0, 25)):
                h = {"split_id": f"split-{rng.randint(0, 3)}", "segment_ord": 0, "doc_id": rng.randint(0, 12)}
                v1 = None if rng.random() < 0.15 else rng.randint(-3, 3)
                h["sort_value"] = None if v1 is None else ("i64", v1)
                if two:
                    v2 = None if rng.random() < 0.2 else rng.randint(0, 2)
                    h["sort_value2"] = None if v2 is None else ("i64", v2)
                hits.append(h)
            # a leaf never reports the same document twice, and reports its hits best first
            uniq = {(h["split_id"], h["doc_id"]): h for h in hits}
            hits = sorted(uniq.values(), key=functools.cmp_to_key(lambda a, b: -better(a, b, o1, o2)))
            for h in hits:
                h["split_id"] = f"{h['split_id']}-leaf{leaf}"   # distinct splits per leaf, like a real fan-out
            nh = len(hits) + rng.randint(0, 50)
            total += nh
            leaves.append(proto.enc_leaf_search_response(nh, hits, num_attempted_splits=1, num_successful_splits=1))
            everything += hits
        sort_fields = [("a", o1)] + ([("b", o2)] if two else [])
        got = proto.dec_leaf_search_response(service.merge_leaf_responses(proto.enc_search_request("{}", max_hits=k, sort_fields=sort_fields), leaves))
        want = sorted(everything, key=functools.cmp_to_key(lambda a, b: -better(a, b, o1, o2)))[:k]
        norm = lambda h: (h["split_id"], h["doc_id"], h.get("sort_value"), h.get("sort_value2") if two else None)
        assert got["num_hits"] == total and [norm(h) for h in got["partial_hits"]] == [norm(h) for h in want], (trial, o1, o2, two, k)


def test_query_ast_compiler_against_a_brute_force_over_documents():
    """QueryAst -> plan (query_compile.cpp: BoolQuery lowering + TantivyBoolQuery::simplify, tantivy_query_ast.rs:166-377;
    bool_query.rs:20-36: a boolean query is a filtering predicate aligned with Elasticsearch) pinned at scale: random
    nested bool / term / range / match_all / match_none trees evaluated document by document in Python, against the
    compiled plan run by the oracle. Doc sets only (no scores)."""
    import random
    rng = random.Random(11)
    vocab = ["red", "green", "blue", "cyan", "pink", "gray"]
    mapping = {"field_mappings": [{"name": "body", "type": "text"}, {"name": "n", "type": "u64", "fast": True}]}
    docs = [{"body": " ".join(rng.sample(vocab, rng.randint(1, 4))), "n": rng.randint(0, 9)} for _ in range(300)]
    img = S.build_split(docs, mapping, "ast-fuzz")
    dm = json.dumps(mapping)

    def gen(depth):
        r = rng.random()
        if depth >= 3 or r < 0.35:
            r = rng.random()
            if r < 0.6:
                return term("body", rng.choice(vocab + ["absent"]))
            if r < 0.85:
                lo, hi = sorted((rng.randint(0, 9), rng.randint(0, 9)))
                return {"type": "range", "field": "n", "lower_bound": {"Included": lo}, "upper_bound": {rng.choice(["Included", "Excluded"]): hi}}
            return {"type": rng.choice(["match_all", "match_none"])}
        q = {"type": "bool"}
        for occur, p in (("must", 0.45), ("should", 0.6), ("must_not", 0.3), ("filter", 0.3)):
            if rng.random() < p:
                q[occur] = [gen(depth + 1) for _ in range(rng.randint(1, 3))]
        if "should" in q and rng.random() < 0.3:
            q["minimum_should_match"] = rng.randint(1, len(q["should"]))
        return q

    def matches(q, d):
        t = q["type"]
        if t == "match_all":
            return True
        if t == "match_none":
            return False
        if t == "term":
            return q["value"] in d["body"].split()
        if t == "range":
            (lk, lv), = q["lower_bound"].items()
            (uk, uv), = q["upper_bound"].items()
            return (d["n"] >= lv if lk == "Included" else d["n"] > lv) and (d["n"] <= uv if uk == "Included" else d["n"] < uv)
        must, should, must_not, flt = q.get("must", []), q.get("should", []), q.get("must_not", []), q.get("filter", [])
        if any(not matches(c, d) for c in must + flt) or any(matches(c, d) for c in must_not):
            return False
        n_should = sum(matches(c, d) for c in should)
        if "minimum_should_match" in q:
            return n_should >= q["minimum_should_match"]
        return n_should >= 1 if (should and not must and not flt) else True

    n_nonempty = 0
    for trial in range(150):
        ast = gen(0)
        want = sorted((i for i, d in enumerate(docs) if matches(ast, d)), reverse=True)
        r = O.split_search(img, service.compile_plan(img, search_request(ast, max_hits=len(docs)), dm))
        assert r.num_hits == len(want) and [h[0] for h in r.hits] == want, (trial, json.dumps(ast), r.num_hits, len(want))
        n_nonempty += bool(want) and len(want) < len(docs)
    assert n_nonempty > 50   # the generator produced discriminating queries, not only all / none


def test_aggregations_end_to_end_against_a_brute_force_over_documents():
    """Leaf aggregation cells -> intermediate bytes -> merge over splits -> finalize (a12, a13/a14, a15) against results
    computed straight from the documents: terms (count-desc / key-asc order, nested stats), histogram (gap filling,
    min_doc_count 0), range buckets, metric aggregations — the Elasticsearch shapes docs/reference/aggregation.md gives
    (`buckets`, `doc_count`, `sum_other_doc_count`, `doc_count_error_upper_bound`, `key`, `from` / `to`, `value`)."""
    import random
    from pipeline import cpu_root_search
    rng = random.Random(23)
    mapping = {"field_mappings": [{"name": "body", "type": "text"}, {"name": "n", "type": "u64", "fast": True},
                                  {"name": "price", "type": "f64", "fast": True}, {"name": "sev", "type": "text", "tokenizer": "raw", "fast": True}]}
    sevs = ["INFO", "WARN", "ERROR", "DEBUG"]
    all_docs = [{"body": rng.choice(["red", "blue"]) + " x", "n": rng.randint(0, 12), "price": rng.randint(0, 400) / 4.0,
                 "sev": rng.choices(sevs, [60, 25, 10, 5])[0]} for _ in range(600)]
    parts = [all_docs[0:250], all_docs[250:420], all_docs[420:600]]
    imgs = [S.build_split(p, mapping, f"agg-fuzz-{i}") for i, p in enumerate(parts)]
    aggs = {
        "by_n": {"terms": {"field": "n", "size": 50}, "aggs": {"p": {"stats": {"field": "price"}}}},
        "by_sev": {"terms": {"field": "sev", "size": 10}},
        "hist": {"histogram": {"field": "price", "interval": 12.5}},
        "ranges": {"range": {"field": "n", "ranges": [{"to": 3}, {"from": 3, "to": 8}, {"from": 8}]}},
        "avg_price": {"avg": {"field": "price"}}, "max_n": {"max": {"field": "n"}}, "cnt": {"value_count": {"field": "n"}},
    }
    for ast, keep in ((MATCH_ALL, lambda d: True), (term("body", "red"), lambda d: d["body"].startswith("red"))):
        got = cpu_root_search(imgs, ast, mapping, max_hits=0, aggs=aggs)["aggregations"]
        docs = [d for d in all_docs if keep(d)]
        # terms on n with nested stats
        by = {}
        for d in docs:
            by.setdefault(d["n"], []).append(d["price"])
        want_terms = sorted(by.items(), key=lambda kv: (-len(kv[1]), kv[0]))
        gb = got["by_n"]["buckets"]
        assert [(b["key"], b["doc_count"]) for b in gb] == [(k, len(v)) for k, v in want_terms]
        assert got["by_n"]["sum_other_doc_count"] == 0 and got["by_n"]["doc_count_error_upper_bound"] == 0
        for b, (k, v) in zip(gb, want_terms):
            st = b["p"]
            assert st["count"] == len(v) and st["min"] == min(v) and st["max"] == max(v)
            assert abs(st["sum"] - sum(v)) < 1e-9 * max(1.0, abs(sum(v))) and abs(st["avg"] - sum(v) / len(v)) < 1e-9 * max(1.0, sum(v) / len(v))
        # terms on a string fast field
        cs = {}
        for d in docs:
            cs[d["sev"]] = cs.get(d["sev"], 0) + 1
        assert [(b["key"], b["doc_count"]) for b in got["by_sev"]["buckets"]] == sorted(cs.items(), key=lambda kv: (-kv[1], kv[0]))
        # histogram: floor(price / interval) * interval, every bucket between the first and the last one present
        hb = {}
        for d in docs:
            k = (d["price"] // 12.5) * 12.5
            hb[k] = hb.get(k, 0) + 1
        lo, hi = min(hb), max(hb)
        want_h = [(lo + 12.5 * i, hb.get(lo + 12.5 * i, 0)) for i in range(int(round((hi - lo) / 12.5)) + 1)]
        assert [(b["key"], b["doc_count"]) for b in got["hist"]["buckets"]] == want_h
        # range buckets: [from, to)
        rb = got["ranges"]["buckets"]
        assert [b["doc_count"] for b in rb] == [sum(d["n"] < 3 for d in docs), sum(3 <= d["n"] < 8 for d in docs), sum(d["n"] >= 8 for d in docs)]
        assert abs(got["avg_price"]["value"] - sum(d["price"] for d in docs) / len(docs)) < 1e-9 * 100
        assert got["max_n"]["value"] == max(d["n"] for d in docs) and got["cnt"]["value"] == len(docs)


def test_bm25_scores_against_a_numpy_restatement_at_corpus_scale():
    """Bm25Weight (tantivy; formula verified against the reference golden in SURVEY.md Appendix B.1) restated in numpy
    float32 from the document lengths and term frequencies themselves: idf = ln(1 + (N - n + 0.5) / (n + 0.5)),
    weight = idf * (1 + k1), norm = k1 * (1 - b + b * fieldnorm / avg_fieldnorm) with the fieldnorm QUANTISED through the
    256-entry id table, score = weight * tf / (tf + norm); a two-term OR adds the contributions in clause order. 4000
    documents of 1..400 tokens (long documents exercise the quantisation) against the oracle's scores, rel. 1e-6
    (logf implementations may differ in the last place; everything else is the same IEEE operations)."""
    import random
    rng = random.Random(5)
    vocab = ["red", "green", "blue"]
    docs = []
    for _ in range(4000):
        n_tok = rng.choice([1, 2, 3, 5, 8, 13, 40, 41, 60, 100, 250, 400])
        toks = [rng.choice(vocab) if rng.random() < 0.3 else "pad" for _ in range(n_tok)]
        docs.append({"body": " ".join(toks)})
    mapping = {"field_mappings": [{"name": "body", "type": "text", "record": "freq", "fieldnorms": True}]}
    img = S.build_split(docs, mapping, "bm25-scale")
    dm = json.dumps(mapping)
    L = ffi.img_lib()
    L.qwgpu_fieldnorm_to_id.restype = C.c_uint8
    L.qwgpu_fieldnorm_to_id.argtypes = [C.c_uint32]
    L.qwgpu_id_to_fieldnorm.restype = C.c_uint32
    L.qwgpu_id_to_fieldnorm.argtypes = [C.c_uint8]
    f32 = np.float32
    lens = np.array([len(d["body"].split()) for d in docs], dtype=np.int64)
    quant = np.array([L.qwgpu_id_to_fieldnorm(L.qwgpu_fieldnorm_to_id(int(x))) for x in lens], dtype=np.float32)
    avg = f32(lens.sum()) / f32(len(docs))
    k1, b = f32(1.2), f32(0.75)
    norm = k1 * (f32(1) - b + b * quant / avg)

    def contributions(word):
        tf = np.array([d["body"].split().count(word) for d in docs], dtype=np.float32)
        n = int((tf > 0).sum())
        idf = np.log(f32(1) + (f32(len(docs) - n) + f32(0.5)) / (f32(n) + f32(0.5)), dtype=np.float32)
        weight = idf * (f32(1) + k1)
        with np.errstate(invalid="ignore"):
            return np.where(tf > 0, weight * (tf / (tf + norm)), f32(0)).astype(np.float32)

    def check(ast, expected):
        r = O.split_search(img, service.compile_plan(img, search_request(ast, max_hits=len(docs), sort_fields=[("_score", DESC)]), dm))
        assert r.num_hits == int((expected > 0).sum())
        got = {h[0]: np.float32(h[4]) for h in r.hits}
        for doc, s in got.items():
            assert abs(float(s) - float(expected[doc])) <= 1e-6 * float(expected[doc]), (doc, float(s), float(expected[doc]))
        # the ranking itself: scores descending, doc id descending among equal scores
        order = [(float(np.float32(h[4])), h[0]) for h in r.hits]
        assert order == sorted(order, key=lambda x: (-x[0], -x[1]))

    check(term("body", "red"), contributions("red"))
    check(bool_(should=[term("body", "red"), term("body", "blue")]), (contributions("red") + contributions("blue")).astype(np.float32))


def test_sort_keys_and_search_after_paging_against_a_python_order():
    """SegmentPartialHitSortingKey (collector.rs:1082-1118: sort value 1, sort value 2 with None last in both
    directions, then doc id in the direction of the first key) and search_after (top_k_collector.rs:821-873) at a
    few hundred documents with missing values: the full order paged K at a time through search_after must equal a
    Python sort of the documents."""
    import functools
    import random
    rng = random.Random(31)
    mapping = {"field_mappings": [{"name": "body", "type": "text"}, {"name": "a", "type": "u64", "fast": True}, {"name": "b", "type": "i64", "fast": True}]}
    docs = []
    for _ in range(400):
        d = {"body": "x"}
        if rng.random() < 0.8:
            d["a"] = rng.randint(0, 6)
        if rng.random() < 0.7:
            d["b"] = rng.randint(-3, 3)
        docs.append(d)
    img = S.build_split(docs, mapping, "sort-page")
    dm = json.dumps(mapping)

    def cmp_opt(x, y, order):
        if x is None or y is None:
            return (x is not None) - (y is not None)
        return ((x > y) - (x < y)) * (1 if order == DESC else -1)

    for o1, o2, two in [(DESC, DESC, True), (ASC, DESC, True), (DESC, ASC, True), (ASC, ASC, False), (DESC, DESC, False)]:
        def better(i, j):
            c = cmp_opt(docs[i].get("a"), docs[j].get("a"), o1)
            if c == 0 and two:
                c = cmp_opt(docs[i].get("b"), docs[j].get("b"), o2)
            if c == 0:
                c = ((i > j) - (i < j)) * (1 if o1 == DESC else -1)
            return c
        want = sorted(range(len(docs)), key=functools.cmp_to_key(lambda i, j: -better(i, j)))
        sort_fields = [("a", o1)] + ([("b", o2)] if two else [])
        got, after, k = [], None, 37
        while True:
            kw = dict(max_hits=k, sort_fields=sort_fields)
            if after is not None:
                kw["search_after"] = after
            resp = proto.dec_leaf_search_response(cpu_split_response_bytes(img, search_request(MATCH_ALL, **kw), dm))
            assert resp["num_hits"] == len(docs)
            page = resp["partial_hits"]
            got += [h["doc_id"] for h in page]
            if len(page) < k:
                break
            after = dict(page[-1])
        assert got == want, (o1, o2, two)


def cpu_split_response_bytes(img, req_pb, dm):
    r = O.split_search(img, service.compile_plan(img, req_pb, dm))
    return service.build_leaf_response(img, req_pb, dm, r.num_hits, r.hits, r.cells)


def test_phrase_queries_against_a_brute_force_over_token_positions():
    """PhraseQuery, slop 0 (full_text mode `phrase`, full_text_query.rs:140-156; tantivy PhraseScorer + Bm25Weight::for_terms):
    a document matches when the words occur at consecutive positions, phrase_count = number of such starts, score =
    (sum of the words' idf) * (1 + k1) * tf_factor(fieldnorm, phrase_count). Documents and counts from a Python scan of
    the token lists, scores from a numpy float32 restatement (rel. 1e-6)."""
    import random
    rng = random.Random(17)
    vocab = ["a", "b", "c", "d"]
    docs = [{"body": " ".join(rng.choice(vocab) for _ in range(rng.choice([2, 3, 5, 9, 20, 45])))} for _ in range(1500)]
    mapping = {"field_mappings": [{"name": "body", "type": "text", "record": "position", "fieldnorms": True}]}
    img = S.build_split(docs, mapping, "phrase-brute")
    dm = json.dumps(mapping)
    L = ffi.img_lib()
    L.qwgpu_fieldnorm_to_id.restype = C.c_uint8
    L.qwgpu_fieldnorm_to_id.argtypes = [C.c_uint32]
    L.qwgpu_id_to_fieldnorm.restype = C.c_uint32
    L.qwgpu_id_to_fieldnorm.argtypes = [C.c_uint8]
    f32 = np.float32
    toks = [d["body"].split() for d in docs]
    lens = np.array([len(t) for t in toks], dtype=np.int64)
    quant = np.array([L.qwgpu_id_to_fieldnorm(L.qwgpu_fieldnorm_to_id(int(x))) for x in lens], dtype=np.float32)
    avg = f32(lens.sum()) / f32(len(docs))
    k1, b = f32(1.2), f32(0.75)
    norm = k1 * (f32(1) - b + b * quant / avg)
    df = {w: sum(w in t for t in toks) for w in vocab}
    idf = lambda w: np.log(f32(1) + (f32(len(docs) - df[w]) + f32(0.5)) / (f32(df[w]) + f32(0.5)), dtype=np.float32)
    for words in (["a", "b"], ["c", "c"], ["a", "b", "c"], ["d", "a", "d"]):
        counts = np.array([sum(t[i:i + len(words)] == words for i in range(len(t) - len(words) + 1)) for t in toks], dtype=np.float32)
        weight = f32(0)
        for w in words:
            weight = weight + idf(w)
        weight = weight * (f32(1) + k1)
        with np.errstate(invalid="ignore"):
            expected = np.where(counts > 0, weight * (counts / (counts + norm)), f32(0)).astype(np.float32)
        ast = {"type": "full_text", "field": "body", "text": " ".join(words), "params": {"mode": {"type": "phrase"}}}
        r = O.split_search(img, service.compile_plan(img, search_request(ast, max_hits=len(docs), sort_fields=[("_score", DESC)]), dm))
        assert r.num_hits == int((counts > 0).sum()) > 0, words
        assert sorted(h[0] for h in r.hits) == [i for i in range(len(docs)) if counts[i] > 0]
        for h in r.hits:
            assert abs(float(np.float32(h[4])) - float(expected[h[0]])) <= 1e-6 * float(expected[h[0]]), (words, h[0])
