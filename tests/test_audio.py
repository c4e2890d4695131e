"""Audio path on the CPU (SURVEY.md 8f-3): the oracle restatement (oracle/ef_oracle_audio.c) against the pins the
unmodified reference produced on its own fixtures (tests/golden/audio_pins.json, tools/make_audio_golden.py) and on
synthetic transport streams (tests/golden/ref_pins.json, tools/make_ref_golden.py), and the constant tables."""
import hashlib
import json
import os

import numpy as np
import pytest

from tests import audio_cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def _masked(pcm, ranges):
    p = pcm.copy()
    for a, b in ranges:
        p[a:b] = 0
    return p


@pytest.mark.parametrize("name", ["splash", "vmedia"])
def test_oracle_matches_reference_pins(oracle, name):
    pins = json.load(open(os.path.join(G, "audio_pins.json")))[name]
    es = oracle.demux_audio_ts(open(os.path.join(G, name + ".ts"), "rb").read())
    assert es.size == pins["es_bytes"] and hashlib.sha256(es.tobytes()).hexdigest() == pins["es_sha256"]
    pcm = oracle.sbc_decode(es)
    assert pcm.size == pins["n_frames"] * 128 and [int(x) for x in pcm[:16]] == pins["pcm_head"]
    assert hashlib.sha256(_masked(pcm, pins["undefined"]).tobytes()).hexdigest() == pins["pcm_sha256_masked"]
    pdm = oracle.pdm(pcm)
    k = pins["pdm_defined_words"]
    assert hashlib.sha256(pdm[:k].tobytes()).hexdigest() == pins["pdm_sha256_defined"]


def test_sbc_tables_match_reference_arrays():
    """espflix_b200/csrc/ef_sbc_tables.h (closed-form matrix, embedded spec window, offsets) against the reference's
    arrays as committed by tools/make_audio_golden.py: SBC_syn_8[i][j] = matrix[i][j]; SBC_proto_8[i][t] = window[t][i]."""
    import re
    g = json.load(open(os.path.join(G, "sbc_tables.json")))
    hdr = open(os.path.join(ROOT, "espflix_b200", "csrc", "ef_sbc_tables.h")).read()

    def table(name):
        i = hdr.index(name)
        return [int(x) for x in re.findall(r"-?\d+", hdr[hdr.index("{", i):hdr.index("};", i)])]

    assert table("ef_sbc_matrix[16][8]") == g["SBC_syn_8"]
    w = np.array(table("ef_sbc_window[10][8]")).reshape(10, 8)
    assert w.T.reshape(-1).tolist() == g["SBC_proto_8"]
    assert table("ef_sbc_offset8[4][8]") == g["SBC_offset8"]


SYNTHETIC_CASES = {"bp28": dict(bitpool=28), "snr_bp12_f0": dict(bitpool=12, allocation=1, frequency=0), "bp60_loud": dict(bitpool=60, loud=True, frequency=3),
                   "rejected_frames": dict(bitpool=28, bad_frames=(3, 4, 17)), "muted_pes": dict(bitpool=28), "pid102": dict(bitpool=28, frequency=1)}


def synthetic_stream(case):
    """(SBC stream, its transport stream) of one synthetic case"""
    es = audio_cases.sbc_stream(1000 + len(case), 40, **SYNTHETIC_CASES[case])
    ts = audio_cases.mux_audio_ts(es, pid=0x102 if case == "pid102" else 0x101, drop_pts_on=(1,) if case == "muted_pes" else ())
    return es, ts


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("case", list(SYNTHETIC_CASES))
def test_oracle_matches_reference_on_synthetic_streams(oracle, case):
    """The reference's demux -> decode_audio -> PDM output on each stream is pinned in tests/golden/ref_pins.json
    (tools/make_ref_golden.py)."""
    pin = json.load(open(os.path.join(G, "ref_pins.json")))["audio"][case]
    es, ts = synthetic_stream(case)
    assert _sha(ts) == pin["in_sha256"], "synthetic stream %s changed" % case
    got_es = oracle.demux_audio_ts(ts)
    assert got_es.size == pin["es_bytes"] and _sha(got_es) == pin["es_sha256"]
    if case == "muted_pes":
        assert got_es.size == es.size - 1024              # the second PES (no PTS) is dropped whole; the third one opens the stream again
    pcm = oracle.sbc_decode(got_es)
    assert pin["pcm_samples"] > 0 and pcm.size == pin["pcm_samples"] and _sha(pcm) == pin["pcm_sha256"]
    pdm = oracle.pdm(pcm)
    assert pdm.size == pin["pdm_words"] and _sha(pdm) == pin["pdm_sha256"]
