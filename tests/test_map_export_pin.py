"""PIN of the C oracle's map export (oracle/lsd_oracle_map.c lsdo_map_export) to lsd_slam_viewer's own KeyFrameDisplay::flushPC
(KeyFrameDisplay.cpp:269-340, compiled unmodified into oracle/_ref/liblsd_ref_viewer.so by oracle/map_oracle.py): every case of
tests/map_export_cases.py -- GT-depth and mapped keyframes, adversarial planes, levels 0-2, five filter settings, three poses
(scale 1, 1.7, 0.35) -- must give the same points, bit for bit.  The viewer library's records are stored in
tests/golden/ref_map_export_320x240.json (tests/golden/make_map_export_golden.py), so this runs on any checkout."""
import json
import os

import numpy as np
import pytest

from oracle import map_oracle
from tests import map_export_cases as mc

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_map_export_320x240.json")


@pytest.fixture(scope="module")
def oracle_records(oracle, seq_small, frames_small):          # `oracle` builds the C oracle that makes the input records
    return mc.pin_records(seq_small, frames_small, False)


def test_oracle_map_export_matches_viewer_records(oracle_records):
    with open(GOLD) as f:
        gold = json.load(f)
    assert set(oracle_records) == set(gold)
    bad = [k for k in gold if oracle_records[k] != gold[k]]
    assert not bad, f"{len(bad)} of {len(gold)} cases differ from the viewer's records, e.g. {bad[:5]}"


def test_cases_cover_the_filter_paths(oracle_records):
    """the stored cases are not vacuous: some keep everything-but-outliers, some keep nothing, NaN records occur"""
    n = {k: v["n"] for k, v in oracle_records.items()}
    assert all(n[f"{name}/L0/F3/P0"] > 0 for name in ("gt", "mapped_kf0", "mapped_kf4", "adversarial"))
    assert any(v == 0 for v in n.values()) or min(n.values()) < max(n.values())
    # the filter depends on the scale: the absolute-variance threshold sees scale^2
    assert all(n[f"{name}/L0/F4/P0"] != n[f"{name}/L0/F4/P1"] for name in ("gt", "mapped_kf0", "mapped_kf4", "adversarial"))


def test_adversarial_planes_reach_the_nan_path(seq_small):
    """var == 0 under a tiny idepth gives depth^4 = inf and 0 * inf = NaN, which passes both thresholds (comparisons with NaN
    are false): the viewer exports such a point, and so must the oracle"""
    idepth, var = mc.adversarial_planes(seq_small.w, seq_small.h, seed=100)
    rec = mc.records_from_planes(idepth, var, np.full(idepth.shape, 128, np.float32))
    pts = map_oracle.map_export(rec, seq_small.w, seq_small.h, mc.level_cam(seq_small.K, 0), mc.POSES[0], 1e-3, 1e-1, 0)
    assert np.isnan(pts[:, :3]).any() and np.isfinite(pts[:, :3]).any()
