#!/usr/bin/env python
"""bench.py — headline benchmark of the per-split leaf-search hot path (BASELINE.json configs[1]).

Workload (config.workload = "c2_bm25_or10_top1000"): BM25 10-term OR query, top-1000 by _score,
over a 100M-doc / 32-split synthetic hdfs-logs-shaped index resident in HBM on each GPU
(3.125M docs per split; body terms with doc-frequency fractions {20,10,5,5,2,2,1,1,0.5,0.1}%).
A "step" = one batch of Q = 4 such queries with DISJOINT term sets (the same 32 splits, different
posting lists), so one step touches Q x postings + the fieldnorm arrays > the 126 MB L2 and the
next step's data has been evicted by then ("inputs larger than L2").

Metric: docs scored per second = postings visited (sum of the query terms' doc frequencies over all
splits) / time. Two timed regions of K steps each (same queries, W warm-up steps before each):
  * `value`: seam C (`qwgpu_split_search`, compiled plans) — device time from CUDA events recorded inside
    libqwgpu on the launching stream around each call's kernel sequence; split data resident in HBM;
  * `e2e`: the reference-facing call `SearchService::leaf_search` = `qwgpu_leaf_search`: host
    LeafSearchRequest protobuf bytes in (QueryAst JSON), host LeafSearchResponse bytes out — request
    decode, plan compilation, H2D of the plans, kernels, D2H of the hits, leaf merge and protobuf
    encoding all inside the wall-clock region.
N > 1: one process per GPU, every rank owns its own 32 splits (weak scaling); in the e2e region ONE
NCCL all-gather of the fixed-size per-rank partial (top-K + counters) per query stands in for the root
merge (`qwgpu_response_to_partial` / `qwgpu_merge_partials`); times are the max over ranks.

`--impl reference`: the reference's CPU algorithm (oracle/qw_oracle.c, a restatement — the real
quickwit-search + tantivy cannot be built here, see DESIGN.md) on all host cores, one split per
thread, on a bounded sample of the same workload.

`--dump-outputs DIR`: what the last timed step of each region returned, as float64 DIR/<name>.npy (rank 0's
view, at most 64 MB in all, a seeded sample of the rows beyond that): split_search_hits (query, split, doc id,
score) and split_search_num_hits[query, split] from `value`; leaf_search_hits (query, split, doc id, sort value)
and leaf_search_num_hits[query] from `e2e`. The inputs are seeded, so two builds run with the same arguments
can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRACS = [0.20, 0.10, 0.05, 0.05, 0.02, 0.02, 0.01, 0.01, 0.005, 0.001]
Q_SETS = 4
K = 1000
# DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) cannot be measured inside the
# timed bench; it is read from profiles/r2_traffic.json, which tools/ncu_traffic.py writes from an
# `ncu --set full` capture of this same command (the capture file is named there).
def ncu_traffic(kernel: str):
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        e = t["kernels"][kernel]
        return float(e["dram_bytes_per_launch"]), f"{t['capture']} ({e['launches']} launches, workload {e['workload']})"
    except Exception:
        return None, None


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="qwgpu", choices=["qwgpu", "reference"])
    ap.add_argument("--splits", type=int, default=32, help="splits per GPU")
    ap.add_argument("--docs-per-split", type=int, default=3_125_000)
    ap.add_argument("--cpu-sample-splits", type=int, default=0, help="splits in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config block (C1 / C3 / C4)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl qwgpu)")
    return a


MSG_VOCAB = 64  # vocabulary of the positions field "msg" (phrase queries of BASELINE config 5)


def build_splits(rank: int, n_splits: int, docs: int, threads: int, msg_vocab: int = 0):
    from quickwit_b200 import splitgen as S

    def one(i):
        gid = rank * n_splits + i
        return S.synth_split(docs, gid, FRACS * Q_SETS, seed=0x5157, ts_start_secs=1_700_000_000 + 86_400 * gid,
                             split_id=f"bench-{gid:04d}", msg_vocab=msg_vocab)
    with ThreadPoolExecutor(max_workers=threads) as ex:
        return list(ex.map(one, range(n_splits)))


def make_plans(imgs):
    """plans[q][s]: 10-term OR, BM25, top-K by _score desc, for query set q on split s."""
    from quickwit_b200 import ffi, plan as P
    plans = []
    for q in range(Q_SETS):
        per_split = []
        for img in imgs:
            root = P.bool_([P.term(img, "body", f"t{q * 10 + i}", occur=ffi.OCCUR_SHOULD) for i in range(10)])
            per_split.append(P.make_plan(root, K, [(ffi.SORT_SCORE, ffi.ORDER_DESC, ffi.ABSENT)]))
        plans.append(per_split)
    return plans


class RawSearch:
    """Pre-marshalled arguments for qwgpu_split_search so the timed region is the C call only."""

    def __init__(self, ctx, split_ids, plans):
        from quickwit_b200 import ffi
        self.L = ffi.lib()
        self.ctx = ctx._ctx
        n = len(split_ids)
        self.n = n
        self.ids = (C.c_char_p * n)(*[s.encode() for s in split_ids])
        self.bufs = [C.create_string_buffer(p, len(p)) for p in plans]
        self.pp = (C.c_void_p * n)(*[C.addressof(b) for b in self.bufs])
        self.ln = (C.c_size_t * n)(*[len(p) for p in plans])
        self.res = (ffi.SplitResult * n)()
        self.status = (C.c_int * n)()
        self.plan_bytes = sum(len(p) for p in plans)

    def run(self):
        rc = self.L.qwgpu_split_search(self.ctx, self.n, self.ids, self.pp, self.ln, self.res, self.status)
        if rc != 0 or any(self.status[i] for i in range(self.n)):
            raise RuntimeError(self.L.qwgpu_last_error().decode())
        r0 = self.res[0]
        out = dict(gpu_us=r0.gpu_time_us, main_us=r0.main_kernel_us, launches=r0.num_kernel_launches,
                   fallbacks=r0.exact_fallbacks,
                   postings=sum(self.res[i].postings_scored for i in range(self.n)),
                   alg_bytes=sum(self.res[i].algorithmic_bytes for i in range(self.n)),
                   hits=sum(self.res[i].num_hits for i in range(self.n)),
                   d2h=sum(32 * self.res[i].num_partial_hits for i in range(self.n)))
        return out

    def partial(self):
        """Fixed-size per-rank partial for the all-gather: merged top-K (score bits, split, doc)."""
        sc = np.concatenate([np.ctypeslib.as_array(C.cast(self.res[i].hits, C.POINTER(C.c_uint64)),
                                                   shape=(self.res[i].num_partial_hits, 4)) for i in range(self.n)
                             if self.res[i].num_partial_hits])
        split = np.concatenate([np.full(self.res[i].num_partial_hits, i, dtype=np.uint64) for i in range(self.n)])
        order = np.lexsort((sc[:, 2] & 0xFFFFFFFF, split, sc[:, 0]))[::-1][:K]
        out = np.zeros((K, 3), dtype=np.uint64)
        out[: len(order), 0] = sc[order, 0]
        out[: len(order), 1] = split[order]
        out[: len(order), 2] = sc[order, 2] & 0xFFFFFFFF
        return out

    def free(self):
        for i in range(self.n):
            self.L.qwgpu_split_result_free(C.byref(self.res[i]))


DUMP_BYTES = 64 << 20  # --dump-outputs writes at most this much in all


def sample_rows(a, max_bytes: int, seed: int = 0):
    """`a` itself if it fits in max_bytes, else a fixed, seeded sample of its rows kept in their order."""
    n = max_bytes // max(1, a[:1].nbytes)
    if len(a) <= n:
        return a
    return a[np.sort(np.random.default_rng(seed).choice(len(a), n, replace=False))]


def split_search_outputs(searches, split_gids):
    """What qwgpu_split_search handed back in each search's latest run, before it is freed: hits rows
    (query, split, doc id, BM25 score) in the order every split returned them, and num_hits[query, split]."""
    rows, num_hits = [], np.zeros((len(searches), len(split_gids)))
    for q, s in enumerate(searches):
        for i in range(s.n):
            r = s.res[i]
            num_hits[q, i] = r.num_hits
            if r.num_partial_hits:  # QwHit as eight u32: v1 (2), v2 (2), doc_id, flags, score (f32), reserved
                h = np.ctypeslib.as_array(C.cast(r.hits, C.POINTER(C.c_uint32)), shape=(r.num_partial_hits, 8))
                rows.append(np.stack([np.full(len(h), q), np.full(len(h), split_gids[i]), h[:, 4], h[:, 6].view(np.float32)], axis=1))
    return (np.concatenate(rows) if rows else np.zeros((0, 4))), num_hits


def leaf_search_outputs(resps, gid_of):
    """The LeafSearchResponse of every query: partial-hit rows (query, split, doc id, sort value) and num_hits[query]."""
    from quickwit_b200 import proto
    rows, num_hits = [], np.zeros(len(resps))
    for q, r in enumerate(resps):
        d = proto.dec_leaf_search_response(r)
        num_hits[q] = d["num_hits"]
        rows += [(q, gid_of[h["split_id"]], h["doc_id"], h.get("sort_value", (None, np.nan))[1]) for h in d["partial_hits"]]
    return np.array(rows, dtype=np.float64).reshape(-1, 4), num_hits


def write_outputs(out_dir: str, arrays: dict):
    os.makedirs(out_dir, exist_ok=True)
    per_array = DUMP_BYTES // len(arrays) - 4096  # (room for the .npy header)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), sample_rows(a, per_array))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def _nvml_loop(self):
        import pynvml as N
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag.is_set():
            try:
                sm = N.nvmlDeviceGetClockInfo(self.handle, N.NVML_CLOCK_SM)
                mask = int(get_reasons(self.handle))
                self.nvml_rows.append((float(sm), [k for k, b in bits.items() if mask & b]))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        # NVML polled every 2 ms (the timed regions last tens of milliseconds); nvidia-smi is the fallback
        self.nvml_rows, self.stop_flag, self.handle = [], threading.Event(), None
        try:
            import pynvml as N
            N.nvmlInit()
            self.handle = N.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml_max = float(N.nvmlDeviceGetMaxClockInfo(self.handle, N.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.handle = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if getattr(self, "handle", None) is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1)
            sm = [r[0] for r in self.nvml_rows]
            reasons = sorted({x for r in self.nvml_rows for x in r[1]})
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.nvml_max, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_oracle_rate(imgs, plans_q0, threads: int, min_seconds: float = 10.0):
    """Times the CPU baseline — oracle/qw_oracle.c's windowed-union / SIMD-unpack organisation of the reference
    algorithm, one (split, query) at a time per C thread (qwo_search_many) — on a bounded sample; postings/s."""
    from oracle import oracle as O
    many = O.ManySearch(imgs, plans_q0)
    many.run(threads)  # warm-up (page in the images)
    t0 = time.perf_counter()
    postings = rounds = 0
    while True:
        postings += many.run(threads)[1]
        rounds += 1
        if time.perf_counter() - t0 >= min_seconds or rounds >= 200:
            break
    dt = time.perf_counter() - t0
    return postings / dt, dt, rounds


T0_SECS = 1_700_000_000
SYNTH_MAPPING = {"field_mappings": [{"name": "body", "type": "text", "record": "freq", "fieldnorms": True},
                                    {"name": "severity_text", "type": "text", "tokenizer": "raw", "fast": True},
                                    {"name": "timestamp", "type": "datetime", "fast": True, "fast_precision": "seconds"},
                                    {"name": "tenant_id", "type": "u64", "fast": True},
                                    {"name": "msg", "type": "text", "record": "position", "fieldnorms": True}], "timestamp_field": "timestamp"}


def other_configs(ctx, imgs, peak, reps: int = 20, lat_runs: int = 60):
    """The other single-GPU BASELINE configs on the same resident index (rank 0, N = 1): device time and
    main-kernel time through seam C (CUDA events inside the library), p50 through qwgpu_leaf_search, and
    the main kernel's roofline fraction from the algorithmic bytes the library accounts per split.
    C1: single term, top-10. C3: term AND timestamp range, top-1000 by timestamp. C4: match_all with
    terms(severity_text) + date_histogram(1h). Units: postings visited (C3: + one column probe each);
    C4: (doc, aggregation) column reads."""
    from quickwit_b200 import proto, service
    n = len(imgs)
    span = 86_400 * n
    term = lambda f, v: {"type": "term", "field": f, "value": v}
    cfgs = {
        "c1_term_top10": (term("severity_text", "ERROR"), dict(max_hits=10), None),
        "c3_term_and_ts_range_top1000_by_ts": ({"type": "bool", "must": [term("body", "t2")]},
                                               dict(max_hits=1000, sort_fields=[("timestamp", 1)], start_timestamp=T0_SECS + span // 4,
                                                    end_timestamp=T0_SECS + 3 * span // 4), None),
        "c4_terms_date_histogram": ({"type": "match_all"}, dict(max_hits=0), C4_AGGS),
    }
    dm = json.dumps(SYNTH_MAPPING)
    ids = [im.split_id for im in imgs]
    offsets = [proto.enc_split_offsets(im.split_id, im.num_docs) for im in imgs]
    out = {}
    for name, (ast, kw, aggs) in cfgs.items():
        sreq = proto.enc_search_request(json.dumps(ast), aggregation_request=json.dumps(aggs) if aggs else None, **kw)
        lreq = proto.enc_leaf_search_request(sreq, offsets, dm)
        plans = [service.compile_plan(im, sreq, dm) for im in imgs]
        rs = RawSearch(ctx, ids, plans)
        for _ in range(3):
            rs.run(); rs.free()
        gpu_us = main_us = 0.0
        for _ in range(reps):
            r = rs.run(); rs.free()
            gpu_us += r["gpu_us"]; main_us += r["main_us"]
        gpu_us /= reps; main_us /= reps
        lat = []
        for i in range(lat_runs + 5):
            t = time.perf_counter()
            resp = ctx.leaf_search(lreq)
            if i >= 5:
                lat.append(time.perf_counter() - t)
        lat.sort()
        dec = proto.dec_leaf_search_response(resp)
        docs = sum(im.num_docs for im in imgs)
        units = r["postings"] if r["postings"] else docs * len(aggs or {})
        achieved = r["alg_bytes"] / main_us / 1e3 if main_us else 0.0
        traffic, tsrc = ncu_traffic(name)
        out[name] = {"value": units / (gpu_us * 1e-6), "unit": "postings/s" if r["postings"] else "column values/s",
                     "num_hits": dec["num_hits"], "device_us": gpu_us, "main_kernel_us": main_us, "launches": r["launches"],
                     "exact_fallbacks": r["fallbacks"], "leaf_search_p50_ms": 1e3 * lat[len(lat) // 2],
                     "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                  "algorithmic_bytes_per_launch": r["alg_bytes"], "traffic": traffic, "traffic_source": tsrc}}
    return out


C4_AGGS = {"by_sev": {"terms": {"field": "severity_text"}},
           "over_time": {"date_histogram": {"field": "timestamp", "fixed_interval": "1h"}}}


def config4_strong(ctx, imgs, world: int, rank: int, reps: int = 10):
    """BASELINE config 4's shape at N > 1 (strong scaling): the 32-split / 100 M-doc corpus sharded over the N
    GPUs (32 / N splits per rank), match_all + terms(severity_text) + date_histogram(1 h), no hits. One
    qwgpu_leaf_search_allgather per query on every rank: the per-rank aggregation partials travel in the
    library's host-staged NCCL all-gather and are merged on every rank. Timed end to end (host bytes in / out),
    barrier on both sides, max over ranks."""
    import torch
    import torch.distributed as dist
    from quickwit_b200 import proto, service
    per = max(1, len(imgs) // world)
    mine = imgs[:per]
    sreq = proto.enc_search_request(json.dumps({"type": "match_all"}), aggregation_request=json.dumps(C4_AGGS), max_hits=0)
    lreq = proto.enc_leaf_search_request(sreq, [proto.enc_split_offsets(im.split_id, im.num_docs) for im in mine], json.dumps(SYNTH_MAPPING))
    got = proto.dec_leaf_search_response(ctx.leaf_search_allgather(lreq))
    # check against the host road: per-rank response -> partial -> torch all-gather -> qwgpu_merge_partials
    nb = service.partial_size(sreq)
    pbuf = torch.zeros(nb, dtype=torch.uint8).pin_memory()
    service.response_to_partial(sreq, ctx.leaf_search(lreq), pbuf.data_ptr(), nb)
    gd = torch.zeros(world * nb, dtype=torch.uint8, device="cuda")
    dist.all_gather_into_tensor(gd, pbuf.cuda())
    gh = gd.cpu()
    want = proto.dec_leaf_search_response(service.merge_partials(sreq, world, gh.data_ptr(), nb))
    assert got["num_hits"] == want["num_hits"] == world * sum(im.num_docs for im in mine)
    assert got["intermediate_aggregation_result"] == want["intermediate_aggregation_result"], "aggregation exchange differs from the host merge"
    for _ in range(3):
        ctx.leaf_search_allgather(lreq)
    torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        ctx.leaf_search_allgather(lreq)
    torch.cuda.synchronize(); dist.barrier()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall = float(t.item()) / reps
    docs = world * sum(im.num_docs for im in mine)
    return {"workload": "c4_terms_date_histogram, corpus sharded over the ranks (strong scaling)", "docs": docs, "splits_per_rank": per,
            "ms_per_query": 1e3 * wall, "docs_per_s": docs / wall, "column_values_per_s": docs * len(C4_AGGS) / wall,
            "api": "qwgpu_leaf_search_allgather (aggregation partials: host-staged NCCL all-gather inside the library)"}


def config2_strong(ctx, imgs, world: int, rank: int, reps: int = 20):
    """The headline query on BASELINE's own index size at N > 1 (strong scaling): the 32-split / 100 M-doc corpus sharded
    over the N GPUs (32 / N splits per rank), BM25 10-term OR, top-1000. One qwgpu_leaf_search_allgather per query on
    every rank (device merge + NCCL all-gather of the per-rank top-K records + device merge of the gathered lists);
    timed end to end with host bytes in / out, barrier on both sides, max over ranks. The merged response of every rank
    is checked against the host road (per-rank response -> partial -> torch all-gather -> qwgpu_merge_partials)."""
    import torch
    import torch.distributed as dist
    from quickwit_b200 import proto, service
    per = max(1, len(imgs) // world)
    mine = imgs[:per]
    sreq = proto.enc_search_request(json.dumps({"type": "bool", "should": [{"type": "term", "field": "body", "value": f"t{i}"} for i in range(10)]}),
                                    max_hits=K, sort_fields=[("_score", 1)])
    lreq = proto.enc_leaf_search_request(sreq, [proto.enc_split_offsets(im.split_id, im.num_docs) for im in mine], json.dumps(SYNTH_MAPPING))
    got = proto.dec_leaf_search_response(ctx.leaf_search_allgather(lreq))
    nb = service.partial_size(sreq)
    pbuf = torch.zeros(nb, dtype=torch.uint8).pin_memory()
    service.response_to_partial(sreq, ctx.leaf_search(lreq), pbuf.data_ptr(), nb)
    gd = torch.zeros(world * nb, dtype=torch.uint8, device="cuda")
    dist.all_gather_into_tensor(gd, pbuf.cuda())
    gh = gd.cpu()
    want = proto.dec_leaf_search_response(service.merge_partials(sreq, world, gh.data_ptr(), nb))
    assert got["num_hits"] == want["num_hits"] and got["partial_hits"] == want["partial_hits"], "cross-rank top-K differs from the host merge"
    from quickwit_b200 import plan as P
    postings = sum(im.doc_freq(P.term(im, "body", f"t{i}").term_ord) for im in mine for i in range(10))
    for _ in range(3):
        ctx.leaf_search_allgather(lreq)
    torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        ctx.leaf_search_allgather(lreq)
    torch.cuda.synchronize(); dist.barrier()
    t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall = float(t.item()) / reps
    c = torch.tensor([postings], dtype=torch.int64, device="cuda")
    dist.all_reduce(c, op=dist.ReduceOp.SUM)
    total = int(c.item())
    return {"workload": "c2_bm25_or10_top1000, corpus sharded over the ranks (strong scaling)", "docs": world * sum(im.num_docs for im in mine),
            "splits_per_rank": per, "ms_per_query": 1e3 * wall, "postings_per_s": total / wall, "postings_per_query": total,
            "api": "qwgpu_leaf_search_allgather (device merge + ncclAllGather of the top-K records + device merge)"}


def config5_mixed(ctx, imgs, peak, world: int, concurrency: int = 64, queries_per_thread: int = 6, announce: bool = False):
    """BASELINE config 5's shape on one GPU's share of the index: a mixed term / phrase / bool / range / aggregation
    query set issued from `concurrency` host threads against the rank's resident splits through qwgpu_leaf_search
    (host protobuf bytes in and out). With N ranks every rank serves its own 32 splits (256 splits / 1 B docs at
    N = 8 with 3.9 M-doc splits; here docs_per_split as configured) — the per-leaf view of a root that fans every
    query out to all leaves — so the job-level QPS is the slowest rank's. Reports QPS, latency percentiles, the mean
    latency per query type and the HBM fraction the mix sustains (algorithmic bytes of the executed queries / wall /
    measured peak). Every response under concurrency is compared with the same request issued alone."""
    import random
    from quickwit_b200 import proto, service
    n = len(imgs)
    span = 86_400 * n
    term = lambda f, v: {"type": "term", "field": f, "value": v}
    or10 = {"type": "bool", "should": [term("body", f"t{i}") for i in range(10)]}
    phrase = lambda text: {"type": "full_text", "field": "msg", "text": text, "params": {"mode": {"type": "phrase"}}}
    mix = [
        ("term_top10", term("severity_text", "ERROR"), dict(max_hits=10), None, 3),
        ("term_bm25_top10", term("body", "t13"), dict(max_hits=10, sort_fields=[("_score", 1)]), None, 2),
        ("phrase_top10", phrase("w1 w2"), dict(max_hits=10, sort_fields=[("_score", 1)]), None, 2),
        ("phrase3_top10", phrase("w0 w3 w1"), dict(max_hits=10, sort_fields=[("_score", 1)]), None, 1),
        ("bool_and_not_top100", {"type": "bool", "must": [term("body", "t0"), term("body", "t1")], "must_not": [term("body", "t4")]},
         dict(max_hits=100, sort_fields=[("tenant_id", 0), ("timestamp", 1)]), None, 2),
        ("range_top1000_by_ts", {"type": "bool", "must": [term("body", "t2")]},
         dict(max_hits=1000, sort_fields=[("timestamp", 1)], start_timestamp=T0_SECS + span // 4, end_timestamp=T0_SECS + 3 * span // 4), None, 2),
        ("or10_bm25_top1000", or10, dict(max_hits=1000, sort_fields=[("_score", 1)]), None, 1),
        ("agg_terms_date_histogram", {"type": "match_all"}, dict(max_hits=0), C4_AGGS, 2),
        ("agg_terms_stats_over_or10", or10, dict(max_hits=0),
         {"tenants": {"terms": {"field": "tenant_id", "size": 10}, "aggs": {"ts": {"stats": {"field": "timestamp"}}}}}, 1),
    ]
    dm = json.dumps(SYNTH_MAPPING)
    ids = [im.split_id for im in imgs]
    offsets = [proto.enc_split_offsets(im.split_id, im.num_docs) for im in imgs]
    reqs, alone, algb, dev_us, weights = {}, {}, {}, {}, []
    for name, ast, kw, aggs, wgt in mix:
        sreq = proto.enc_search_request(json.dumps(ast), aggregation_request=json.dumps(aggs) if aggs else None, **kw)
        reqs[name] = proto.enc_leaf_search_request(sreq, offsets, dm)
        rs = RawSearch(ctx, ids, [service.compile_plan(im, sreq, dm) for im in imgs])
        for _ in range(2):
            r = rs.run(); rs.free()
        algb[name] = r["alg_bytes"]
        dev_us[name] = r["gpu_us"]
        for _ in range(2):
            alone[name] = ctx.leaf_search(reqs[name])
        weights += [name] * wgt
    rng = random.Random(5)
    plan = [[rng.choice(weights) for _ in range(queries_per_thread)] for _ in range(concurrency)]
    lat, got = [[] for _ in range(concurrency)], [[] for _ in range(concurrency)]
    start = threading.Barrier(concurrency + 1)

    errs = []

    def worker(t):
        # untimed warm-up: the thread's whole plan once, so that every in-flight call slot of the library (stream,
        # pinned staging, device scratch: allocated on first use, grown to the largest request seen) exists
        try:
            for name in plan[t]:
                ctx.leaf_search(reqs[name])
        except Exception as e:  # noqa: BLE001  (reported after the join; the barrier below must still be reached)
            errs.append(e)
        try:
            start.wait(timeout=600)
        except threading.BrokenBarrierError:
            return
        if errs:
            return
        try:
            for name in plan[t]:
                if announce:  # (with QWGPU_TRACE=1: labels the library's per-call phase timings on stderr)
                    print(f"[c5] {name}", file=sys.stderr, flush=True)
                t0 = time.perf_counter()
                resp = ctx.leaf_search(reqs[name])
                lat[t].append((name, time.perf_counter() - t0))
                got[t].append((name, resp))
        except Exception as e:  # noqa: BLE001
            errs.append(e)
    ths = [threading.Thread(target=worker, args=(t,)) for t in range(concurrency)]
    for th in ths:
        th.start()
    start.wait(timeout=600)
    t0 = time.perf_counter()
    for th in ths:
        th.join()
    wall = time.perf_counter() - t0
    if errs:
        raise RuntimeError(f"config 5: {len(errs)} worker(s) failed, first: {errs[0]}")
    # outside the timed region: every response (distinct byte strings decoded once) against the sequential one
    key = lambda r: (lambda d: (d["num_hits"], d["partial_hits"], d["intermediate_aggregation_result"]))(proto.dec_leaf_search_response(r))
    want = {name: key(r) for name, r in alone.items()}
    seen = {(name, resp) for g in got for name, resp in g}
    mismatches = sorted({name for name, resp in seen if key(resp) != want[name]})
    if mismatches:
        raise RuntimeError(f"config 5: responses under concurrency differ from the sequential ones: {mismatches}")
    flat = sorted(x for l in lat for _, x in l)
    per_type = {}
    for l in lat:
        for name, x in l:
            per_type.setdefault(name, []).append(x)
    nq = len(flat)
    bytes_total = sum(algb[name] for l in lat for name, _ in l)
    pct = lambda q: 1e3 * flat[min(nq - 1, int(q * nq))]
    return {"workload": "c5_mixed_term_phrase_bool_range_agg", "concurrency": concurrency, "queries": nq,
            "splits_per_gpu": n, "docs_per_gpu": sum(im.num_docs for im in imgs), "n_gpus": world,
            "qps": nq / wall, "latency_ms": {"p50": pct(0.50), "p90": pct(0.90), "p99": pct(0.99), "max": 1e3 * flat[-1]},
            "mean_latency_ms_by_type": {k: 1e3 * sum(v) / len(v) for k, v in sorted(per_type.items())},
            "device_us_alone_by_type": dev_us, "mix_weights": {m[0]: m[4] for m in mix},
            "hbm": {"algorithmic_bytes": bytes_total, "achieved_gbs": bytes_total / wall / 1e9, "peak": peak, "frac": bytes_total / wall / 1e9 / peak},
            "api": "qwgpu_leaf_search from 64 host threads; responses checked against the sequential ones"}


def main():
    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    import __graft_entry__ as g
    if not os.path.exists(os.path.join(ROOT, "quickwit_b200", "libqwgpu.so")):
        g.build()

    workload = {"workload": "c2_bm25_or10_top1000", "splits_per_gpu": a.splits, "docs_per_split": a.docs_per_split,
                "docs_per_gpu": a.splits * a.docs_per_split, "queries_per_step": Q_SETS, "top_k": K,
                "term_df_fractions": FRACS, "l2": "inputs larger than L2 (disjoint term sets per query in a step)"}

    if a.impl == "reference":
        # the reference's CPU algorithm on the host cores; rank 0 only
        if rank != 0:
            return
        n_s = a.cpu_sample_splits or min(a.splits, max(4, min(cores, 32)))
        threads = min(cores, Q_SETS * n_s, 256)  # every (query set, split) pair is a task: all the host threads there is work for
        imgs = build_splits(0, n_s, a.docs_per_split, threads=min(cores, 32))
        plans = make_plans(imgs)
        from oracle import oracle as O
        many = O.ManySearch([imgs[i] for q in range(Q_SETS) for i in range(n_s)], [plans[q][i] for q in range(Q_SETS) for i in range(n_s)])
        times, postings_step = [], 0
        for s in range(a.warmup + a.steps):
            t0 = time.perf_counter()
            postings_step = many.run(threads)[1]
            dt = time.perf_counter() - t0
            if s >= a.warmup:
                times.append(dt)
        total = sum(times)
        value = postings_step * len(times) / total
        sample = f"{Q_SETS} queries x {n_s} of {a.splits} splits ({n_s * a.docs_per_split} docs) per step, {threads} C threads, windowed union + SIMD unpack"
        print(json.dumps({"impl": "reference", "metric": "docs_scored_per_sec", "value": value, "unit": "postings/s",
                          "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * total / len(times),
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+u32",
                          "data": "synthetic", "config": workload,
                          "cpu_baseline": {"value": value, "unit": "postings/s", "cores": threads, "kind": "port", "sample": sample},
                          "e2e": {"value": value, "unit": "postings/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # stdout carries exactly one JSON line: anything libraries print meanwhile (NCCL's version banner
    # goes to stdout) is sent to stderr, and the result is written to the saved descriptor at the end
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from quickwit_b200.service import SearcherContext

    t_build = time.perf_counter()
    imgs = build_splits(rank, a.splits, a.docs_per_split, threads=max(1, min(cores // max(world, 1), 32)),
                        msg_vocab=0 if a.no_configs else MSG_VOCAB)
    plans = make_plans(imgs)
    ctx = SearcherContext(local_rank)
    for img in imgs:
        ctx.register_split(img)
    resident = ctx.resident_bytes()
    ids = [im.split_id for im in imgs]
    searches = [RawSearch(ctx, ids, plans[q]) for q in range(Q_SETS)]
    # the same queries as LeafSearchRequest protobufs (QueryAst JSON), for the e2e region
    from quickwit_b200 import proto, service
    doc_mapper = json.dumps({"field_mappings": [{"name": "body", "type": "text", "record": "freq", "fieldnorms": True},
                                                {"name": "timestamp", "type": "datetime", "fast": True}], "timestamp_field": "timestamp"})
    offsets = [proto.enc_split_offsets(im.split_id, im.num_docs) for im in imgs]
    sreqs = [proto.enc_search_request(json.dumps({"type": "bool", "should": [{"type": "term", "field": "body", "value": f"t{q * 10 + i}"} for i in range(10)]}),
                                      max_hits=K, sort_fields=[("_score", 1)]) for q in range(Q_SETS)]
    lreqs = [proto.enc_leaf_search_request(sr, offsets, doc_mapper) for sr in sreqs]
    t_build = time.perf_counter() - t_build
    part_bytes = service.partial_size(sreqs[0]) if world > 1 else 0
    device_exchange = world > 1 and not os.environ.get("QWGPU_HOST_EXCHANGE")
    if device_exchange:
        # the library's own collective: NCCL communicator per context + the global split table
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(SearcherContext.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        all_ids = [f"bench-{g:04d}" for g in range(world * a.splits)]
        ctx.comm_init(bytes(uid.cpu().numpy().tobytes()), rank, world, all_ids)
        # one communicator ("lane") per concurrent query of a step: query q of every step runs on lane q on every
        # rank, so each communicator sees its collectives in the same order everywhere
        for lane in range(1, Q_SETS):
            if rank == 0:
                uid.copy_(torch.frombuffer(bytearray(SearcherContext.comm_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            ctx.comm_init_lane(lane, bytes(uid.cpu().numpy().tobytes()), rank, world)
    if world > 1 and not device_exchange:
        # one fixed-size partial per query of the step; the step's partials travel in ONE all-gather
        part_host = torch.zeros(Q_SETS * part_bytes, dtype=torch.uint8).pin_memory()
        part_dev = torch.zeros(Q_SETS * part_bytes, dtype=torch.uint8, device="cuda")
        gath_dev = torch.zeros(world * Q_SETS * part_bytes, dtype=torch.uint8, device="cuda")
        gath_host = torch.zeros(world * Q_SETS * part_bytes, dtype=torch.uint8).pin_memory()
        by_query = torch.zeros(Q_SETS * world * part_bytes, dtype=torch.uint8)  # [query][rank][partial]

    def step(keep: bool = False):
        acc = dict(gpu_us=0.0, main_us=0.0, launches=0, postings=0, alg_bytes=0, d2h=0, h2d=0, fallbacks=0)
        for s in searches:
            r = s.run()
            acc["gpu_us"] += r["gpu_us"]
            acc["main_us"] += r["main_us"]
            for k in ("launches", "postings", "alg_bytes", "d2h", "fallbacks"):
                acc[k] += r[k]
            acc["h2d"] += s.plan_bytes
            if not keep:
                s.free()
        return acc

    last = {}

    # The step's queries are issued concurrently, one host thread per query, like concurrent searches on
    # a searcher node (the library is thread-safe: one stream + staging slot per in-flight call). The
    # window kernels still run one after the other on the device — each fills every SM — so this only
    # overlaps one query's host work (plan compile, response merge / encode) with another's kernels.
    pool = ThreadPoolExecutor(max_workers=Q_SETS)
    lat = []

    def one_query(q):
        t = time.perf_counter()
        r = ctx.leaf_search(lreqs[q])
        lat.append(time.perf_counter() - t)
        if world > 1 and not device_exchange:  # this rank's merged leaf response -> fixed-size partial (typed sort values, split id, doc id)
            service.response_to_partial(sreqs[q], r, part_host.data_ptr() + q * part_bytes, part_bytes)
        return r

    def merge_query(q):
        return service.merge_partials(sreqs[q], world, by_query.data_ptr() + q * world * part_bytes, part_bytes)

    phase = [0.0, 0.0, 0.0]  # leaf searches, all-gather round trip, root merges (rank-local wall time)

    def step_e2e():
        t0 = time.perf_counter()
        if device_exchange:
            # the step's queries run concurrently, query q on communicator lane q (a communicator's collectives are
            # issued in the same order on every rank); the search, the NCCL all-gather of the per-rank records and
            # the cross-rank merge all run inside qwgpu_leaf_search_allgather on the call's stream (no host bounce,
            # no Python in between)
            def one_collective(q):
                t = time.perf_counter()
                r = ctx.leaf_search_allgather(lreqs[q], lane=q)
                lat.append(time.perf_counter() - t)
                return r
            resps = list(pool.map(one_collective, range(Q_SETS)))
            phase[0] += time.perf_counter() - t0
        else:
            resps = list(pool.map(one_query, range(Q_SETS)))
            phase[0] += time.perf_counter() - t0
        if world > 1 and not device_exchange:
            t0 = time.perf_counter()
            part_dev.copy_(part_host, non_blocking=True)
            dist.all_gather_into_tensor(gath_dev, part_dev)   # the single collective of the data path
            gath_host.copy_(gath_dev)
            # [rank][query][partial] -> [query][rank][partial], then every rank runs the root merge
            by_query.view(Q_SETS, world, part_bytes).copy_(gath_host.view(world, Q_SETS, part_bytes).transpose(0, 1))
            phase[1] += time.perf_counter() - t0
            t0 = time.perf_counter()
            resps = list(pool.map(merge_query, range(Q_SETS)))
            phase[2] += time.perf_counter() - t0
        for q in range(Q_SETS):
            last[q] = resps[q]

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    if device_exchange:
        # correctness of the device-side exchange, once, outside the timed regions: the same query through the
        # host path (per-rank response -> fixed-size partial -> all-gather -> qwgpu_merge_partials)
        pb = torch.zeros(part_bytes, dtype=torch.uint8).pin_memory()
        service.response_to_partial(sreqs[0], ctx.leaf_search(lreqs[0]), pb.data_ptr(), part_bytes)
        gd = torch.zeros(world * part_bytes, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(gd, pb.cuda())
        gh = gd.cpu()
        want = proto.dec_leaf_search_response(service.merge_partials(sreqs[0], world, gh.data_ptr(), part_bytes))
        got = proto.dec_leaf_search_response(ctx.leaf_search_allgather(lreqs[0]))
        assert got["num_hits"] == want["num_hits"] and got["partial_hits"] == want["partial_hits"], "device-side exchange differs from the host merge"
        assert got["num_attempted_splits"] == want["num_attempted_splits"] == world * a.splits
    for _ in range(max(a.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    sync()
    t0 = time.perf_counter()
    # the last timed step's results are freed after the clock stops, so that --dump-outputs reads them
    # without a copy inside the timed region
    accs = [step(keep=i == a.steps - 1) for i in range(a.steps)]
    sync()
    wall_c = time.perf_counter() - t0
    gids = [rank * a.splits + i for i in range(a.splits)]
    split_out = split_search_outputs(searches, gids) if a.dump_outputs and rank == 0 else None
    for s in searches:
        s.free()
    for _ in range(max(a.warmup, 3)):
        step_e2e()
    sync()
    lat.clear()
    phase[:] = [0.0, 0.0, 0.0]
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step_e2e()
    sync()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    # latency of ONE query in flight (SURVEY.md §8d: >= 200 timed runs after 20 warm-ups, index resident),
    # outside the timed regions; plus the cost of making one cold split resident (image H2D + tables)
    single = []
    if rank == 0:
        for i in range(220):
            t = time.perf_counter()
            ctx.leaf_search(lreqs[i % Q_SETS])
            if i >= 20:
                single.append(time.perf_counter() - t)
        single.sort()
        t = time.perf_counter()
        ctx.unregister_split(imgs[-1].split_id)
        ctx.register_split(imgs[-1])
        cold_ms = 1e3 * (time.perf_counter() - t)
    hits0 = proto.dec_leaf_search_response(last[0])
    assert len(hits0["partial_hits"]) == K and hits0["num_hits"] > 0
    if split_out is not None:
        leaf_out = leaf_search_outputs([last[q] for q in range(Q_SETS)], {f"bench-{g:04d}": g for g in range(world * a.splits)})
        write_outputs(a.dump_outputs, {"split_search_hits": split_out[0], "split_search_num_hits": split_out[1],
                                       "leaf_search_hits": leaf_out[0], "leaf_search_num_hits": leaf_out[1]})

    gpu_s = sum(x["gpu_us"] for x in accs) * 1e-6
    main_s = sum(x["main_us"] for x in accs) * 1e-6
    postings = sum(x["postings"] for x in accs)
    alg_bytes = sum(x["alg_bytes"] for x in accs)
    launches = sum(x["launches"] for x in accs)
    n_main = a.steps * Q_SETS
    postings_rank0 = postings
    c4_strong = None
    c2_strong = None
    if world > 1 and device_exchange and not a.no_configs and a.splits % world == 0:
        try:
            c4_strong = config4_strong(ctx, imgs, world, rank)
        except AssertionError as e:  # (the same data on every rank: a mismatch shows on all of them)
            c4_strong = {"error": str(e)}
        try:
            c2_strong = config2_strong(ctx, imgs, world, rank)
        except AssertionError as e:
            c2_strong = {"error": str(e)}
    # BASELINE config 5's shape (mixed query set, concurrency 64) on every rank's share of the index; the job-level
    # figures are the slowest rank's
    c5 = None
    if not a.no_configs:
        peak5 = 6650.0
        try:
            peak5 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
        except Exception:
            pass
        if world > 1:
            dist.barrier()
        # (an auxiliary block must never cost the headline line: a failure is reported in place of the block, and at
        # N > 1 every rank still takes part in the reduction)
        try:
            c5 = config5_mixed(ctx, imgs, peak5, world)
        except Exception as e:  # noqa: BLE001
            c5 = {"error": f"{type(e).__name__}: {e}"[:500]}
        if world > 1:
            bad = "error" in c5
            v = torch.tensor([1.0 if bad else 0.0] + ([0.0] * 6 if bad else [-c5["qps"], c5["latency_ms"]["p50"], c5["latency_ms"]["p90"], c5["latency_ms"]["p99"],
                                                                          c5["latency_ms"]["max"], -c5["hbm"]["frac"]]), dtype=torch.float64, device="cuda")
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
            anybad, q, p50, p90, p99, mx, fr = [float(x) for x in v.tolist()]
            if anybad:
                c5 = c5 if bad else {"error": "config 5 failed on another rank"}
            else:
                c5["qps"] = -q
                c5["latency_ms"] = {"p50": p50, "p90": p90, "p99": p99, "max": mx}
                c5["hbm"]["frac"] = -fr
                c5["aggregate"] = "slowest rank (every query is answered by every rank's leaf)"
    if world > 1:
        t = torch.tensor([gpu_s, wall, main_s, wall_c], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gpu_s, wall, main_s, wall_c = [float(x) for x in t.tolist()]
        c = torch.tensor([postings, launches], dtype=torch.int64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        postings, launches = [int(x) for x in c.tolist()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = (alg_bytes / n_main) / (main_s / n_main) / 1e9 if main_s > 0 else 0.0  # rank-0 kernel
    out = {
        "metric": "docs_scored_per_sec", "value": postings / gpu_s, "unit": "postings/s", "n_gpus": world,
        "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": 1e3 * gpu_s / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+u32", "data": "synthetic",
        "config": workload,
        "setup": {"parallelism": f"splits_x{world}", "resident_bytes_per_gpu": resident, "build_seconds": round(t_build, 1)},
        "e2e": {"value": postings / wall, "unit": "postings/s", "api": "qwgpu_leaf_search (LeafSearchRequest -> LeafSearchResponse bytes)",
                "ms_per_step": 1e3 * wall / a.steps, "concurrent_queries": Q_SETS,
                "single_query_latency_ms": {"p50": 1e3 * single[len(single) // 2], "p90": 1e3 * single[int(len(single) * 0.9)],
                                            "p99": 1e3 * single[int(len(single) * 0.99)], "runs": len(single)},
                "exchange": ("device: qwgpu_leaf_search_allgather (NCCL all-gather + merge inside the library)" if device_exchange else ("host partials" if world > 1 else None)),
                "cold_split_register_ms": cold_ms, "phase_ms_per_step": {"leaf_search": 1e3 * phase[0] / a.steps, "all_gather": 1e3 * phase[1] / a.steps, "root_merge": 1e3 * phase[2] / a.steps}, "mean_query_latency_ms": 1e3 * sum(lat) / max(len(lat), 1),
                "h2d_bytes_per_step": accs[0]["h2d"] + sum(len(x) for x in lreqs),
                "d2h_bytes_per_step": Q_SETS * (a.splits * 32 + 64 + 40 * K),  # per split 32 B of counters + the merged top-K record (device merge)
                "seam_c_wall_value": postings / wall_c},
        "gpu_launches": launches,
        "exact_fallbacks": sum(x["fallbacks"] for x in accs),
        "roofline": {"bound": "hbm", "kernel": "k_union<COLLECT>", "achieved": achieved, "peak": peak,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                     "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic("k_union<COLLECT>")[0] if (a.splits, a.docs_per_split) == (32, 3_125_000) else None,
                     "traffic_source": ncu_traffic("k_union<COLLECT>")[1],
                     "algorithmic_bytes_per_launch": alg_bytes / n_main, "avg_launch_us": 1e6 * main_s / n_main},
        "clocks": clocks,
    }
    if world == 1 and not a.no_configs:
        try:
            out["configs"] = other_configs(ctx, imgs, peak)
        except Exception as e:  # noqa: BLE001  (auxiliary block: reported, never fatal for the line)
            out["configs"] = {"error": f"{type(e).__name__}: {e}"[:500]}
    if c4_strong:
        out["config4_strong"] = c4_strong
    if c2_strong:
        out["config2_strong"] = c2_strong
    if c5:
        out["config5_mixed"] = c5
    if not a.no_cpu_baseline and world == 1:
        n_s = a.cpu_sample_splits or min(a.splits, max(4, min(cores, 32)))
        threads = min(cores, Q_SETS * n_s, 256)
        rate, dt, rounds = cpu_oracle_rate([imgs[i] for q in range(Q_SETS) for i in range(n_s)], [plans[q][i] for q in range(Q_SETS) for i in range(n_s)], threads)
        out["cpu_baseline"] = {"value": rate, "unit": "postings/s", "cores": threads, "kind": "port",
                               "sample": f"{Q_SETS} query sets over {n_s} splits ({Q_SETS * n_s} tasks) x {rounds} rounds ({dt:.1f} s), {threads} C threads, windowed union + SIMD unpack"}
    sys.stdout.flush()
    os.write(result_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
