"""Pins the C restatement (oracle/tsdr_oracle.c) to the REAL reference.

Every scenario below runs a stage of an oracle on seeded inputs and lists what it observed.  The reference's own list --
made by the compiled reference (oracle/_ref, built from the original sources) running the same scenario -- is stored in
tests/golden/reference_outputs.json (tests/golden/make_reference_outputs.py), arrays as digests of their bits; the
restatement has to reproduce it bit for bit.  tests/golden/*.npz pin a few paths with the arrays themselves.

CPU only; no GPU, no product code.
"""
import numpy as np
import pytest

from oracle import oracle as orc
from tempestsdr_b200 import synth
from tests.test_golden import assert_matches_reference

CFGS = {  # name: (samplerate, height, refreshrate)
    "cfg1": (8_000_000, 525, 60.0),
    "cfg2": (25_000_000, 1125, 60.0),
    "cfg5": (50_000_000, 1125, 60.0),
    "exact2": (1_000_000, 100, 50.0),    # r == 2.0 exactly: the reference leaves one stale pixel per block
    "odd": (2_400_000, 313, 59.94),
}

SCENARIOS = {}


def scenario(fn):
    """Registers fn(O, **params) -> [(label, value)] for make_reference_outputs.py."""
    SCENARIOS[fn.__name__] = fn
    return fn


def key(fn_name, /, **params):
    return f"oracle_pinning/{fn_name}" + "".join(f"/{k}={v}" for k, v in sorted(params.items()))


def check(fn, /, **params):
    assert_matches_reference(key(fn.__name__, **params), fn(orc.port(), **params))


@scenario
def am_demod(O):
    iq = synth.noise_iq(50_001, seed=1)
    iq[:8] = [0, 0, 1e-30, 1e-30, 3e38, 1e38, -0.0, 0.0]
    return [("am_demod", O.am_demod(iq)), ("empty", O.am_demod(np.zeros(0, np.float32)).size)]


def test_am_demod():
    check(am_demod)


@scenario
def resample_stream(O, name, nearest):
    fs, h, fv = CFGS[name]
    w, _, _ = O.geometry(fs, h, fv)
    obs = [("geometry", O.geometry(fs, h, fv))]
    block = int(0.1 * fs / fv)
    rng = np.random.default_rng(7)
    rs = O.resampler()
    up = w * h * fv
    # r == 2 exactly: the reference's loop emits one pixel fewer than it sizes the buffer for (dsp.c:262 vs
    # :288-297), so the last slot keeps what an earlier call left there -- zero while the buffer never moves,
    # uninitialised heap once a ragged block makes it grow.  Equal blocks are compared whole; with ragged blocks
    # the one undefined slot is excluded.
    stale_tail = (name == "exact2") and not nearest
    for ragged in (False, True):
        for k in range(14):
            n = block if (k % 5 or not ragged) else max(3, block // 3 + k)
            x = rng.uniform(0, 1, n).astype(np.float32)
            a = rs.run(x, up, fs, nearest)
            if stale_tail and ragged:
                if O.kind == "port":
                    assert rs.last_emitted == a.size - 1
                a = a[:-1]
            obs += [(f"resample {name} ragged={ragged} block {k}", a), (f"state after block {k}", rs.state)]
    return obs


@pytest.mark.parametrize("name", list(CFGS))
@pytest.mark.parametrize("nearest", [False, True])
def test_resample_stream(name, nearest):
    check(resample_stream, name=name, nearest=nearest)


@scenario
def resample_general_ratio(O, ratio):
    rng = np.random.default_rng(11)
    rs, lead = O.resampler(), orc.port().resampler()
    obs = []
    for k in range(9):
        x = rng.standard_normal(1000 + 37 * k).astype(np.float32)
        a = rs.run(x, ratio * 1e6, 1e6)
        lead.run(x, ratio * 1e6, 1e6)
        # when (size-offset)*r lands exactly on an integer the loop writes one pixel fewer than output_samples and,
        # the buffer having grown, the reference's last slot is uninitialised heap: exclude exactly that slot (the
        # restatement, run in step, tells how many pixels the loop wrote)
        obs += [(f"ratio {ratio} block {k}", a[:min(lead.last_emitted, a.size)]), (f"state after block {k}", rs.state)]
    return obs


@pytest.mark.parametrize("ratio", [0.37, 0.9999, 1.0, 1.5, 2.0, 3.25])
def test_resample_general_ratio(ratio):
    check(resample_general_ratio, ratio=ratio)


@scenario
def dropcomp(O):
    rng = np.random.default_rng(3)
    obs = []
    for i in range(400):
        block = int(rng.integers(1, 5000))
        diff = int(rng.integers(0, 3 * block))
        off = int(rng.integers(-4 * block, 4 * block))
        size = int(rng.integers(0, 4 * block))
        obs += [(f"{i} shift_with", O.dropcomp_shift_with(diff, block, off)),
                (f"{i} will_drop_all", O.dropcomp_will_drop_all(diff, size, block))]
        obs += [(f"{i} add ring_accepts={ok}", O.dropcomp_add(diff, size, block, ok)) for ok in (True, False)]
    return obs


def test_dropcomp():
    check(dropcomp)


@scenario
def frame_stage_pieces(O):
    w, h = 507, 525
    f = synth.video_like_frame(w, h, seed=5, shift_x=100, shift_y=40)
    f[1234] = 512.0; f[99] = -300.0     # marker values must pass through auto-gain
    obs = []
    st = orc.Autogain(0, 0, 1)
    for k in range(3):
        obs += [(f"autogain {k}", O.autogain(st, f, 0.1)), (f"autogain state {k}", (st.lastmax, st.lastmin, st.snr))]
    s = np.zeros(w * h, np.float32)
    for c in (0.0, 0.3, 0.97):
        O.timelowpass(c, f, s)
        obs.append((f"timelowpass {c}", s.copy()))
    wa, ha = O.average_v_h(f, w, h)
    obs += [("colsum", wa), ("rowsum", ha)]
    for n in (1, 2, 3, 4, 5, 6, 17, 507):
        s = np.random.default_rng(n).uniform(0, 5, n).astype(np.float32)
        obs.append((f"gauss n={n}", O.gaussianblur(s)))
    for strip in (wa, ha):
        for size in (5, 13, strip.size // 3):
            obs.append((f"findbestfit {strip.size} {size}", O.findbestfit(strip, float(strip.sum()), size)))
    sw = orc.Sweetspot()
    for k in range(6):
        o = O.findthesweetspot(sw, np.roll(wa, 17 * k), int(w * 0.05), 0.9)
        obs += [(f"sweetspot state {k}", sw.astuple()), (f"sweetspot strip {k}", o)]
    return obs


def test_frame_stage_pieces():
    check(frame_stage_pieces)


PP_FIELDS = ("avg_speed", "pll_state", "lastmax", "lastmin", "refreshrate_after", "width_after", "pll_callback_fired",
             "autogain_callback_fired", "autogain_cb_min", "autogain_cb_max", "snr")


@scenario
def post_process_sequence(O, lpbs, aap, autoshift, pll, mb):
    fs, hgt, fv = CFGS["cfg1"]
    pp = O.postprocessor(fs, hgt, fv, autoshift, pll)
    w, _, _ = O.geometry(fs, hgt, fv)
    obs = []
    for k in range(9):
        f = synth.video_like_frame(w, hgt, seed=k, shift_x=60 + 9 * k, shift_y=20 + 3 * k)
        a, r = pp.run(f, w, hgt, mb, 0.1, lpbs, aap)
        obs += [(f"frame {k}", a), (f"sync {k}", (r.x.astuple(), r.y.astuple()))]
        obs += [(f"{fld} {k}", getattr(r, fld)) for fld in PP_FIELDS]
    return obs


@pytest.mark.parametrize("lpbs,aap,autoshift,pll,mb", [
    (1, 0, 1, 0, 0.0),   # GUI default minus PLL
    (1, 0, 1, 1, 0.0),   # GUI default
    (1, 1, 1, 0, 0.4),
    (0, 0, 1, 0, 0.3),
    (0, 1, 0, 0, 0.0),   # green marker lines drawn into the input buffer
    (0, 0, 0, 0, 0.5),
    (1, 0, 0, 0, 0.0),   # green lines on a copy
])
def test_post_process_sequence(lpbs, aap, autoshift, pll, mb):
    check(post_process_sequence, lpbs=lpbs, aap=aap, autoshift=autoshift, pll=pll, mb=mb)


@scenario
def post_process_resize_and_flag_flip(O):
    pp = O.postprocessor(8_000_000, 525, 60.0)
    shapes = [(200, 100, 1), (200, 100, 1), (150, 120, 1), (150, 120, 0), (300, 200, 0), (200, 100, 1)]
    obs = []
    for k, (w, h, lpbs) in enumerate(shapes):
        f = synth.video_like_frame(w, h, seed=40 + k, shift_x=11, shift_y=7)
        obs.append((f"resize step {k}", pp.run(f, w, h, 0.25, 0.1, lpbs, 0)[0]))
    return obs


def test_post_process_resize_and_flag_flip():
    check(post_process_resize_and_flag_flip)


@scenario
def fft(O, logn):
    x = synth.noise_iq(1 << logn, seed=logn)
    return [(f"fft 2^{logn} inv={inv}", O.fft(x, inv)) for inv in (False, True)]


@pytest.mark.parametrize("logn", [0, 1, 2, 3, 7, 12, 16])
def test_fft(logn):
    check(fft, logn=logn)


@scenario
def autocorrelation_and_xcorr(O, size):
    x = np.abs(synth.noise_iq(size, seed=size)[:size])
    obs = [("autocorrelation", O.autocorrelation(x))]
    if size >= 4:
        a = synth.noise_iq(size, seed=1); b = synth.noise_iq(size, seed=2)
        n = orc.port().fft_getrealsize(size)
        obs.append(("xcorr", O.crosscorrelation(a, b)[: 2 * n]))
    return obs


@pytest.mark.parametrize("size", [1, 5, 1000, 4096, 70_001])
def test_autocorrelation_and_xcorr(size):
    check(autocorrelation_and_xcorr, size=size)


@scenario
def framerate_detector_plots(O):
    P = orc.port()                 # the capture size and the demodulated input come from the restatement (pinned above)
    fs = 2_000_000
    size = P.framerate_capture_size(fs)
    det = O.framerate_detector()
    obs = []
    for k in range(3):
        x = P.am_demod(synth.video_like_iq(size, fs, 400, 200, 50.0, seed=k))
        (fo, fp), (lo, lp), c = det.run(fs, x)
        assert c == k + 1
        if O.kind == "port":
            assert P.framerate_windows(fs) == (fo, fo + fp.size, lo, lo + lp.size)
        obs += [(f"offsets and calls {k}", (fo, lo, c)), (f"frame plot {k}", fp), (f"line plot {k}", lp)]
    return obs


def test_framerate_detector_plots():
    check(framerate_detector_plots)


@scenario
def superbandwidth_stitch(O):
    fs, fv = 400_000, 50.0
    sif = int(fs / fv)             # 8000 samples per frame, does not divide 2^k
    pairs = 10 * sif               # 80000 -> N = 65536
    base = synth.video_like_iq(pairs + 5000, fs, 200, 160, fv, seed=9, snr_db=25)
    hops = []
    for i, lag in enumerate((0, 1234, 77, 3999)):
        seg = base[2 * lag: 2 * (lag + pairs)].copy()
        seg += synth.noise_iq(pairs, seed=100 + i, scale=0.01)
        hops.append(seg)
    n2 = 2 * orc.port().fft_getrealsize(pairs)
    obs = [(f"bestfit hop {i}", O.superb_bestfit(hops[0][:n2], hops[i][:n2], sif)) for i in range(1, 4)]
    obs.append(("abs diff", O.complex_to_abs_diff(hops[1][:4096])))
    out, offs = O.superb_ondataready(hops, sif)
    return obs + [("offsets", list(offs)), ("stitched", out)]


def test_superbandwidth_stitch():
    check(superbandwidth_stitch)


def test_pixel_rule():
    P = orc.port()
    f = np.array([-1, 0, 1e-9, 0.5, 1.0, 1.0001, 256, 512, 1024, 2048, 7], dtype=np.float32)
    g = int(0.5 * 255.0)
    assert list(P.pixels_argb(f)) == [0, 0, 0, g | g << 8 | g << 16, 0xFFFFFF, 0xFFFFFF, 255 << 16, 255 << 8, 255, 0, 0xFFFFFF]
    assert list(P.pixels_argb(f, True))[:5] == [0xFFFFFF, 0xFFFFFF, 0xFFFFFF, (255 - g) * 0x010101, 0]
