#!/usr/bin/env python3
"""tools/make_ref_golden.py — pins of the UNMODIFIED reference (oracle/_ref: decoder CLI, composite / pacing library,
index builder, audio CLI) on the synthetic and random inputs of the oracle-vs-reference tests, so that those tests
run wherever the repository is checked out. Writes tests/golden/ref_pins.json:

  decode        per coverage stream (tests/synth_cases.py): SHA-256 of the TS and of every picture efref_decode emits
  video         per composite case of tests/test_oracle_vs_ref.py: SHA-256 of the input frame and of the field / blit
  presentation  the same for the _hscroll / overlay / progress / fade cases
  index         make_index() tables of fuzzed streams and the video.idx image of three of them (tests/test_tsindex.py)
  audio         demux -> decode_audio -> PDM of the synthetic SBC streams (tests/test_audio.py): sizes and SHA-256
  pacing        irregular PTS lists with the flip list and poster scroll push_video / video_isr produced for them

The inputs come from the tests' own case lists (the pacing lists are stored whole); build oracle/_ref first
(oracle/Makefile, target ref)."""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import oracle_lib  # noqa: E402
from tests import test_audio, test_oracle_vs_ref, test_tsindex  # noqa: E402
from tests.synth_cases import COVERAGE  # noqa: E402

sha256 = test_oracle_vs_ref.sha256


def decode_pins():
    pins = {}
    for idx, (name, kw) in enumerate(COVERAGE):
        _, ts = test_oracle_vs_ref.coverage_ts(idx)
        info, frames = oracle_lib.ref_decode_ts(ts)
        assert info["frames"] == frames.shape[0] == kw["n_pictures"], name
        pins[name] = {"in_sha256": sha256(ts), "frames": int(info["frames"]), "frame_sha256": [sha256(f) for f in frames]}
    return pins


def case_pins(rv, cases):
    return {key: {"in_sha256": sha256(*test_oracle_vs_ref.case_inputs(args)), "out_sha256": sha256(getattr(rv, method)(*args))}
            for key, method, args in cases()}


def index_pins():
    ri = oracle_lib.RefIndexer()
    tables = {}
    for seed in test_tsindex.FUZZ_TABLE_SEEDS:
        ts = test_tsindex.fuzz_table_ts(seed)
        r = ri.make_index(ts)
        tables[str(seed)] = {"in_sha256": hashlib.sha256(ts).hexdigest(), "first_pts": r["first_pts"], "last_pts": r["last_pts"],
                             "seq_pts": [int(x) for x in r["seq_pts"]], "seq_pos": [int(x) for x in r["seq_pos"]]}
    files = test_tsindex.fuzz_image_files()
    img = ri.build_idx(files)
    return {"tables": tables, "image": {"in_sha256": hashlib.sha256(b"".join(files)).hexdigest(), "bytes": len(img), "sha256": hashlib.sha256(img).hexdigest()}}


def audio_pins():
    pins = {}
    for case in test_audio.SYNTHETIC_CASES:
        _, ts = test_audio.synthetic_stream(case)
        with tempfile.TemporaryDirectory() as d:
            p, out = os.path.join(d, "a.ts"), os.path.join(d, "a.bin")
            open(p, "wb").write(ts.tobytes())
            subprocess.run([os.path.join(ROOT, "oracle", "_ref", "efref_audio"), p, out], check=True, capture_output=True, timeout=120)   # one process per run: the reference keeps its state in globals
            raw = open(out, "rb").read()
        nes, npcm = [int(x) for x in np.frombuffer(raw[:16], dtype=np.uint64)]
        es = np.frombuffer(raw[16:16 + nes], dtype=np.uint8)
        pcm = np.frombuffer(raw[16 + nes:16 + nes + 2 * npcm], dtype=np.int16)
        pdm = np.frombuffer(raw[16 + nes + 2 * npcm:], dtype=np.uint16)
        pins[case] = {"in_sha256": sha256(ts), "es_bytes": int(es.size), "es_sha256": sha256(es), "pcm_samples": int(pcm.size), "pcm_sha256": sha256(pcm),
                      "pdm_words": int(pdm.size), "pdm_sha256": sha256(pdm)}
    return pins


def pacing_pins(rv):
    """Jitter, repeated and decreasing PTS (late frames, 'resetting v timing'), long gaps, both standards."""
    rng = np.random.default_rng(2024)
    frames = np.zeros((2, 101376), dtype=np.uint8)                      # content is irrelevant to the schedule
    cases = []
    for case in range(24):
        ntsc = case % 2
        n = int(rng.integers(2, 14))
        step = rng.choice([3003, 3003, 3003, 1501, 6006, 0, -4000, 45045], size=n)
        pts = (129003 + np.cumsum(step)).astype(np.int64)
        pts = np.maximum(pts, 0)
        fc0 = int(rng.integers(0, 4)) if case < 8 else int(rng.integers(1, 100000))
        fr = np.ascontiguousarray(np.broadcast_to(frames[0], (n, 101376)))
        modes = np.where(rng.random(n) < 0.2, rng.integers(1, 4, size=n), 0).astype(np.int32)      # 1 at once, 2 / 3 poster scroll
        tail = int(rng.integers(0, 20))
        f, ff, fl, _, hs = rv.paced(fr, pts, ntsc, fc0, 400, want_fields=False, modes=modes, tail_fields=tail, want_hscroll=True)
        cases.append({"ntsc": ntsc, "pts": [int(x) for x in pts], "frame_counter0": fc0, "max_fields": 400, "modes": [int(x) for x in modes],
                      "tail_fields": tail, "fields": f, "flip_field": [int(x) for x in ff], "flip_line": [int(x) for x in fl], "hscroll": [int(x) for x in hs]})
    return cases


def main():
    if not (oracle_lib.have_ref() and oracle_lib.have_ref_index()):
        raise SystemExit("oracle/_ref is not built: make -C oracle ref")
    rv = oracle_lib.RefVideo()
    pins = {"decode": decode_pins(), "video": case_pins(rv, test_oracle_vs_ref.video_cases),
            "presentation": case_pins(rv, test_oracle_vs_ref.presentation_cases), "index": index_pins(), "audio": audio_pins(),
            "pacing": pacing_pins(rv)}
    path = os.path.join(ROOT, "tests", "golden", "ref_pins.json")
    with open(path, "w") as f:
        json.dump(pins, f, indent=1)
        f.write("\n")
    print(path, os.path.getsize(path), "bytes;", {k: len(v) for k, v in pins.items()})


if __name__ == "__main__":
    main()
