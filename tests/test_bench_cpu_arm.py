"""CPU tier: the two CPU implementations bench.py's reference arm times -- the oracle port (oracle_frame) and the reference's own source
as far as it compiles here (reference_frame over oracle/_ref) -- do the same work on the same frame: identical numbers of matches from
both projection searches (the reference arm reports the faster of the two, so they must be interchangeable)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import pyoracle as po  # noqa: E402

needs_ref = pytest.mark.skipif(not bench.reference_source_available(), reason="oracle/_ref is not built and no reference checkout is given")


@needs_ref
def test_reference_source_frame_equals_the_oracle_frame():
    c = bench.CONFIGS[3]
    pairs = bench.make_pairs(2, c["W"], c["H"], base=4)
    for i in range(2):
        eL, eR = po.OracleExtractor(c["NFEAT"], 1.2, 8, 20, 7), po.OracleExtractor(c["NFEAT"], 1.2, 8, 20, 7)
        rL, rR = po.RefExtractor(c["NFEAT"], 1.2, 8, 20, 7), po.RefExtractor(c["NFEAT"], 1.2, 8, 20, 7)
        o = bench.oracle_frame(pairs[i, 0], pairs[i, 1], eL, eR, c["cam"], c["W"], c["H"])
        n = bench.reference_frame(pairs[i, 0], pairs[i, 1], rL, rR, c["cam"], c["W"], c["H"])
        assert n == int((o["fm"] >= 0).sum()) + int((o["mt"] >= 0).sum()) and n > 1000


@needs_ref
def test_threaded_drivers_run():
    c = bench.CONFIGS[3]
    pairs = bench.make_pairs(4, c["W"], c["H"], base=4)
    r1, _ = bench.cpu_oracle_frames(pairs, 4)
    r2, _ = bench.cpu_reference_frames(pairs, 4)
    assert r1 > 0 and r2 > 0


def test_issue_table_is_the_ratio_it_claims():
    import json
    cnt = json.load(open(os.path.join(ROOT, "profiles", "r02_inst_counts.json")))
    t = bench.issue_table({"fast": 0.423, "blur": 0.264, "pyramid": 0.188, "orient_desc": 0.153, "quadtree": 0.25}, 128, 1965, cnt)
    f = t["stages"]["fast"]["warp_inst_per_clk_per_sm"]
    assert abs(f - 371081902 / (0.423e-3 * 1965e6 * 148)) < 1e-9 and 2.9 < f < 3.1
    assert 1.9 < t["stages"]["blur"]["warp_inst_per_clk_per_sm"] < 2.1            # at the half-rate pipe's limit
    assert "quadtree" not in t["stages"] and bench.issue_table({"fast": 0.4}, 128, None, cnt)["stages"] == {}
    half = bench.issue_table({"fast": 0.423}, 64, 1965, cnt)["stages"]["fast"]["warp_inst_per_clk_per_sm"]
    assert abs(half - f / 2) < 1e-9                                                # counts scale with the images of a launch
