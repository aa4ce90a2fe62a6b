"""Golden vectors captured from the REAL reference (tests/golden/make_golden.py) checked against
  * the C restatement  (CPU, always), and
  * the CUDA path      (tests/test_gpu_parity.py reuses `load` from here on the GPU box).

The scenario tests that compare with the reference (test_oracle_pinning, test_host_library, test_rawfile_plugin) read what
the reference returned from tests/golden/reference_outputs.json (tests/golden/make_reference_outputs.py): scalars as they
are, arrays as a digest of their bits (`observed`), so that a bit-exact comparison needs no stored array.
"""
import hashlib
import json
import math
import os

import numpy as np
import pytest

from oracle import oracle as orc
from tempestsdr_b200 import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
REFERENCE_OUTPUTS = os.path.join(GOLD, "reference_outputs.json")


def load(name):
    return np.load(os.path.join(GOLD, name))


def observed(v):
    """A JSON-comparable form of what a scenario observed: arrays become dtype, shape and a SHA-256 of their bits (equal
    digests mean bit-identical arrays), tuples become lists, bytes become text, NaN becomes the string "nan"."""
    if isinstance(v, np.ndarray):
        a = np.ascontiguousarray(v)
        return f"{a.dtype.str}{list(a.shape)}:{hashlib.sha256(a.tobytes()).hexdigest()[:32]}"
    if isinstance(v, (list, tuple)):
        return [observed(x) for x in v]
    if isinstance(v, bytes):
        return v.decode("latin-1")
    if isinstance(v, np.generic):
        v = v.item()
    if isinstance(v, float) and math.isnan(v):
        return "nan"
    return v


def reference_outputs(key):
    """What the compiled reference returned in scenario `key`, as recorded by make_reference_outputs.py."""
    with open(REFERENCE_OUTPUTS) as f:
        return json.load(f)[key]


def assert_matches_reference(key, observations):
    """`observations`: (label, value) pairs from one scenario run against this project's code; compared one by one with the
    reference's values for the same scenario."""
    want = reference_outputs(key)
    got = [(label, observed(v)) for label, v in observations]
    assert len(got) == len(want), f"{key}: {len(got)} observations, the reference made {len(want)}"
    bad = [(label, g, w) for (label, g), w in zip(got, want) if g != w]
    assert not bad, f"{key}: {len(bad)} of {len(got)} differ from the reference, first: {bad[0]}"


def same_bits(a, b):
    a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
    v = np.uint32 if a.dtype == np.float32 else np.uint64
    return a.shape == b.shape and np.array_equal(a.view(v), b.view(v))


def test_golden_demod_resample():
    g = load("demod_resample.npz")
    P = orc.port()
    fs, h, fv, w, block = int(g["fs"]), int(g["h"]), float(g["fv"]), int(g["w"]), int(g["block"])
    iq = synth.video_like_iq(6 * block, fs, 2 * w // 2, h, fv, seed=int(g["seed"]))
    mag = P.am_demod(iq)
    assert same_bits(mag, g["mag"])
    for nn, key in ((False, "pixels"), (True, "pixels_nn")):
        rs = P.resampler()
        pix = [rs.run(mag[k * block:(k + 1) * block], w * h * fv, fs, nn) for k in range(6)]
        assert [p.size for p in pix] == list(g["counts"])
        assert same_bits(np.concatenate(pix), g[key])
        if not nn:
            assert rs.state == tuple(g["states"][-1])


@pytest.mark.parametrize("name,mb,lpbs,aap,sx,sy", [("frame_stage_default.npz", 0.0, 1, 0, (31, 5), (11, 1)),
                                                   ("frame_stage_blur.npz", 0.35, 0, 1, (40, 0), (9, 0))])
def test_golden_frame_stage(name, mb, lpbs, aap, sx, sy):
    g = load(name)
    P = orc.port()
    w, h = int(g["w"]), int(g["h"])
    pp = P.postprocessor(800_000, 105, 60.0, autoshift=1, pll=0)
    for k, seed in enumerate(g["seeds"]):
        f = synth.video_like_frame(w, h, seed=int(seed), shift_x=sx[0] + sx[1] * k, shift_y=sy[0] + sy[1] * k)
        o, res = pp.run(f, w, h, mb, 0.1, lpbs, aap)
        assert same_bits(o, g["out"][k]), f"frame {k}"
        assert [res.x.dx, res.x.vx, res.x.curr_stripsize, res.y.dx, res.y.vx, res.y.curr_stripsize] == list(g["meta"][k])


def test_golden_fft_autocorr():
    P = orc.port()
    g = load("fft_4096.npz")
    assert same_bits(P.fft(g["x"], False), g["fwd"]) and same_bits(P.fft(g["x"], True), g["inv"])
    g = load("autocorr_20000.npz")
    assert same_bits(P.autocorrelation(g["x"]), g["ac"])
    g = load("framerate_plots.npz")
    det = P.framerate_detector()
    for s in g["seeds"]:
        c = P.am_demod(synth.video_like_iq(int(g["size"]), int(g["fs"]), 300, 120, 55.5, seed=int(s)))
        (fo, fp), (lo, lp), calls = det.run(int(g["fs"]), c)
    assert (fo, lo) == (int(g["frame_off"]), int(g["line_off"]))
    assert same_bits(fp, g["frame_plot"]) and same_bits(lp, g["line_plot"])


def superb_hops(g):
    sif, pairs = int(g["sif"]), int(g["pairs"])
    base = synth.video_like_iq(pairs + 3000, int(g["fs"]), 100, 80, float(g["fv"]), seed=9, snr_db=25)
    return [base[2 * l: 2 * (l + pairs)].copy() + synth.noise_iq(pairs, seed=100 + i, scale=0.01)
            for i, l in enumerate(g["lags"])], sif


def test_golden_superbandwidth():
    g = load("superb_4x16384.npz")
    hops, sif = superb_hops(g)
    out, offs = orc.port().superb_ondataready(hops, sif)
    assert list(offs) == list(g["offsets"])
    assert same_bits(out, g["out"])
