"""PTS -> field pacing of push_video (SURVEY.md 8f-2; video.cpp:1023-1057, 1165-1177), CPU side: the C restatement
of the schedule against the pins the unmodified reference produced (tools/make_pacing_golden.py), and against what
the reference itself (real push_video / video_isr on two threads) produced for irregular PTS (tools/make_ref_golden.py)."""
import json
import os

import numpy as np
import pytest

from tests.oracle_lib import Oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PINS = json.load(open(os.path.join(ROOT, "tests", "golden", "pacing_pins.json")))


@pytest.mark.parametrize("name", sorted(PINS))
def test_schedule_matches_reference_pins(name):
    p = PINS[name]
    pts = 129003 + 3003 * np.arange(p["pictures"], dtype=np.int64)
    fields, ff, fl, hs = Oracle().paced_schedule(pts, p["ntsc"], p["frame_counter0"], p["max_fields"], modes=p["modes"], tail_fields=p["tail_fields"], want_hscroll=True)
    assert fields == p["fields"] and ff.tolist() == p["flip_field"] and fl.tolist() == p["flip_line"]
    assert hs.tolist() == p["hscroll"]                    # the poster scroll (_animate / _easd) field by field


def test_schedule_matches_reference_on_irregular_pts():
    """Jitter, repeated and decreasing PTS (late frames, 'resetting v timing'), long gaps, both standards: the
    schedules the reference's real push_video / video_isr produced for these PTS lists, pinned with them in
    tests/golden/ref_pins.json (tools/make_ref_golden.py)."""
    o = Oracle()
    cases = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_pins.json")))["pacing"]
    assert len(cases) == 24
    for case, p in enumerate(cases):
        pts = np.array(p["pts"], dtype=np.int64)
        f, ff, fl, hs = o.paced_schedule(pts, p["ntsc"], p["frame_counter0"], p["max_fields"], modes=p["modes"], tail_fields=p["tail_fields"], want_hscroll=True)
        assert (f, ff.tolist(), fl.tolist()) == (p["fields"], p["flip_field"], p["flip_line"]), (case, p["ntsc"], p["frame_counter0"], p["pts"])
        assert hs.tolist() == p["hscroll"], (case, p["modes"])
