"""Writes tests/golden/ref_map_export_320x240.json: the records of the map-export cases (tests/map_export_cases.py) computed by
oracle/_ref/liblsd_ref_viewer.so, i.e. by lsd_slam_viewer's own KeyFrameDisplay::setFrom / refreshPC / flushPC compiled unmodified
(oracle/map_oracle.py).  Each record is the number of points and the SHA-256 of their bytes; tests/test_map_export_pin.py holds
the C oracle's lsdo_map_export to them.  Needs the reference sources to build oracle/_ref.  Leaves every other golden file alone.
Run:  python -m tests.golden.make_map_export_golden
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "ref_map_export_320x240.json")

if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    from lsd_slam_b200 import synth
    from oracle import map_oracle, pyoracle
    from tests import map_export_cases as mc
    pyoracle.build()
    if not map_oracle.viewer_available():
        raise SystemExit("the reference viewer sources are absent: the viewer's records cannot be regenerated")
    map_oracle.build()
    seq = synth.Sequence(320, 240, seed=1234)
    frames = {k: seq.render(k) for k in range(0, 8)}
    recs = mc.pin_records(seq, frames, "ref_viewer")
    with open(OUT, "w") as f:
        json.dump(recs, f, indent=1, sort_keys=True)
    print(f"{len(recs)} cases, {sum(r['n'] for r in recs.values())} points")
