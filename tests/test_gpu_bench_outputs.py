"""bench.py --dump-outputs: the arrays it writes are what the timed searches returned (checked against the CPU
oracle on the same seeded splits), and a second run with the same arguments writes the same arrays."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPLITS, DOCS = 2, 50_000
NAMES = {"split_search_hits", "split_search_num_hits", "leaf_search_hits", "leaf_search_num_hits"}


def _dump(out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--splits", str(SPLITS),
                        "--docs-per-split", str(DOCS), "--no-configs", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert len([l for l in r.stdout.splitlines() if l.strip()]) == 1
    assert {f[:-4] for f in os.listdir(out)} == NAMES
    return {n: np.load(out / f"{n}.npy") for n in NAMES}


def test_dumped_outputs_match_the_oracle_and_repeat(tmp_path):
    got = _dump(tmp_path / "a")
    assert all(a.dtype == np.float64 for a in got.values())
    imgs = bench.build_splits(0, SPLITS, DOCS, threads=SPLITS)
    plans = bench.make_plans(imgs)
    hits, nh, leaf_hits = got["split_search_hits"], got["split_search_num_hits"], got["leaf_search_hits"]
    assert nh.shape == (bench.Q_SETS, SPLITS)
    for q in range(bench.Q_SETS):
        for s, img in enumerate(imgs):
            want = O.split_search(img, plans[q][s])
            mine = hits[(hits[:, 0] == q) & (hits[:, 1] == s)]
            assert nh[q, s] == want.num_hits
            assert mine[:, 2].tolist() == [h[0] for h in want.hits]
            assert np.array_equal(mine[:, 3].astype(np.float32), np.array([h[4] for h in want.hits], dtype=np.float32))
        # the e2e region's response to the same query: the hit count over the splits and the K best of their scores
        leaf = leaf_hits[leaf_hits[:, 0] == q]
        assert got["leaf_search_num_hits"][q] == nh[q].sum()
        assert len(leaf) == bench.K
        best = np.sort(hits[hits[:, 0] == q, 3].astype(np.float32))[::-1][:bench.K]
        assert np.array_equal(np.sort(leaf[:, 3].astype(np.float32))[::-1], best)
    again = _dump(tmp_path / "b")
    for name in NAMES:
        assert np.array_equal(got[name], again[name]), name
