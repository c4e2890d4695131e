"""The oracle restatement against the UNMODIFIED reference on the synthetic coverage streams and on random
frames, plus assertions that those streams really exercise the paths the reference's fixtures lack. The
reference's outputs are pinned in tests/golden/ref_pins.json (tools/make_ref_golden.py runs the reference on
the inputs the case lists below produce); every pin also holds a digest of its input, so a changed input
generator is reported as such and not as a wrong output."""
import hashlib
import json
import os

import numpy as np
import pytest

from espflix_b200 import synth
from tests.synth_cases import COVERAGE, make

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def pins(section):
    return json.load(open(os.path.join(ROOT, "tests", "golden", "ref_pins.json")))[section]


def sha256(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def coverage_ts(idx):
    name, kw = COVERAGE[idx]
    es, off = make(idx, kw)
    return es, synth.wrap_ts(es, off)


def video_cases():
    """(key, method, args) of the composite comparisons: Oracle and oracle_lib.RefVideo share these methods."""
    rng = np.random.default_rng(7)
    for ntsc in (1, 0):
        for fc in (0, 1, 2):
            fr = rng.integers(0, 249, 101376, dtype=np.uint8)
            yield "field:%d:%d" % (ntsc, fc), "field", (fr, ntsc, fc)
        fr = rng.integers(0, 256, 101376, dtype=np.uint8)          # bytes above 248: dither carries cross bytes
        yield "field:%d:1:carry" % ntsc, "field", (fr, ntsc, 1)
        for line, x, w in ((0, 0, 352), (191, 0, 352), (77, 16, 64), (100, 8, 344)):
            yield "blit:%d:%d:%d:%d" % (ntsc, line, x, w), "blit", (fr, ntsc, line, x, w, 1)


PRESENTATION_CASES = [(0, 0, 0), (8, 0, 0), (-8, 0, 0), (176, 0, 0), (-344, 0, 0), (344, -1, 100), (0, 32, 0), (0, 5, 239), (0, 31, 17), (24, 1, 300)]


def presentation_cases():
    """SURVEY.md 8f-2: _hscroll two-frame scroll and the composite() overlay / progress bar / fade."""
    rng = np.random.default_rng(11)
    a, b = rng.integers(0, 249, 101376, dtype=np.uint8), rng.integers(0, 249, 101376, dtype=np.uint8)
    bm = rng.integers(0, 256, 1280, dtype=np.uint8)
    for ntsc in (1, 0):
        for hs, blend, prog in PRESENTATION_CASES:
            yield "field_ex:%d:%d:%d:%d" % (ntsc, hs, blend, prog), "field_ex", (a, b, ntsc, 1, hs, bm, blend, prog)


def case_inputs(args):
    return [a for a in args if isinstance(a, np.ndarray)]


def _check_cases(oracle, section, cases):
    want = pins(section)
    assert sorted(want) == sorted(key for key, _, _ in cases())
    for key, method, args in cases():
        assert sha256(*case_inputs(args)) == want[key]["in_sha256"], "input of %s changed" % key
        assert sha256(getattr(oracle, method)(*args)) == want[key]["out_sha256"], key


@pytest.mark.parametrize("idx", range(len(COVERAGE)), ids=[c[0] for c in COVERAGE])
def test_port_equals_reference_on_synthetic(oracle, idx):
    name, kw = COVERAGE[idx]
    es, ts = coverage_ts(idx)
    pin = pins("decode")[name]
    assert sha256(ts) == pin["in_sha256"], "synthetic stream %s changed" % name
    got = oracle.decode_ts(ts)
    assert pin["frames"] == kw["n_pictures"] == got.shape[0]
    assert [sha256(f) for f in got] == pin["frame_sha256"], name
    assert [sha256(f) for f in oracle.decode_es(es)] == pin["frame_sha256"], "ES path"
    assert np.array_equal(oracle.demux_ts(ts), es), "TS wrapper round trip"


def test_coverage_set_reaches_the_missing_paths(oracle):
    oracle.stats_reset()
    for idx, (name, kw) in enumerate(COVERAGE):
        oracle.decode_es(make(idx, kw)[0])
    s = oracle.stats()
    t = list(s.mb_type)
    assert t[0x11] > 0 and t[0x12] > 0 and t[0x1A] > 0, "macroblock-level quantiser changes"
    assert t[0x01] > 0 and t[0x02] > 0 and t[0x08] > 0 and t[0x0A] > 0
    assert s.full_pel_mbs > 0
    assert s.f_code[3] > 0 and s.f_code[1] > 0
    assert s.escapes16 > 0
    assert s.q2_zero > 0, "quirk Q2 (zero coefficient becomes +1)"
    assert all(v > 0 for v in s.mocomp_xy), "all four half-pel cases"
    assert s.skipped > 0 and s.blocks_dc_only > 0
    assert s.pictures[1] > 0 and s.pictures[2] > 0
    assert s.pin_out_of_domain == 0, "coverage streams must stay inside the reference's defined clamp domain"


def test_reference_video_equals_port_on_random_frames(oracle):
    _check_cases(oracle, "video", video_cases)


def test_presentation_extras_port_equals_reference(oracle):
    _check_cases(oracle, "presentation", presentation_cases)
