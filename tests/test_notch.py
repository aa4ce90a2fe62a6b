"""The notch filter and the power spectrum (csrc/notch.cu): filter design, its frequency response and the configuration rules on
the host; the kernels against float64 models, block-cut behaviour, the pipeline as the composition "notch, then the un-notched
pipeline", the in-band-carrier use case, live reconfiguration, superbandwidth mode and the host library's TSDR_NOTCH and
TSDR_SPECTRUM knobs."""
import ctypes as C
import threading
import time

import numpy as np
import pytest
import scipy.signal

from tempestsdr_b200 import _native
from tests.test_tuner import _collect_pipeline, _same, cplx, emitter, iq, raster_corr, OWN_MIN

BETA = 0.1102 * (80.0 - 8.7)
DK = (80.0 - 7.95) / (2.285 * 2.0 * np.pi)


def delta(fs, L):
    return DK * fs / (L - 1)


def design(fs, centers, widths, ntaps=0):
    lib = _native.lib()
    c = np.ascontiguousarray(centers, np.float64)
    w = np.ascontiguousarray(widths, np.float64)
    taps = np.zeros(2 * 8193, np.float32)
    n, nfft = C.c_int(0), C.c_int(0)
    rc = lib.tsdrgpu_notch_design(fs, c.size, c.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p), ntaps,
                                  taps.ctypes.data_as(C.c_void_p), 8193, C.byref(n), C.byref(nfft))
    return rc, taps[: 2 * n.value].view(np.complex64), nfft.value


def numpy_design(fs, centers, widths, L):
    """The definition restated: h[n] = delta[n - c] - sum_j firwin(L, w_j / 2, kaiser)[n] e^{2 pi i f_j (n - c) / fs}."""
    c = (L - 1) // 2
    m = np.arange(L) - c
    h = np.zeros(L, np.complex128)
    h[c] = 1.0
    for f, w in zip(centers, widths):
        g = scipy.signal.firwin(L, w / 2, window=("kaiser", BETA), fs=fs)
        h -= g * np.exp(2j * np.pi * f * m / fs)
    return h


CONFIGS = [(10_000_000, [1e6, -2e6], [200e3, 100e3], 0),
           (8_000_000, [-3.85e6, 0.0, 1.5e6], [100e3, 40e3, 300e3], 0),
           (100_000_000, list(np.linspace(-40e6, 40e6, 32)), [1e6] * 32, 0),
           (2_000_000, [0.0], [10e3], 0),
           (25_000_000, [1e6, 1.3e6, 1.6e6], [100e3, 100e3, 100e3], 8193),
           (8_000_000, [2e6], [1.4e6], 65),
           (48_000, [-20_000.0, 5_000.0], [6_000.0, 4_000.0], 129)]


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("fs,centers,widths,ntaps", CONFIGS)
def test_design_matches_the_definition(fs, centers, widths, ntaps):
    rc, taps, nfft = design(fs, centers, widths, ntaps)
    assert rc == 0, _native.lib().tsdrgpu_last_error(None)
    want = numpy_design(fs, centers, widths, taps.size)
    assert np.max(np.abs(taps.astype(np.complex128) - want)) <= 1e-7


@pytest.mark.parametrize("fs,centers,widths,ntaps", CONFIGS)
def test_frequency_response_bounds(fs, centers, widths, ntaps):
    """The float32 taps' DTFT: |H| <= 2e-4 over every notch's core [f - w/2 + delta/2, f + w/2 - delta/2] (the 80 dB design's
    1e-4 ripple with a factor 2 for Kaiser's width estimate and the float32 rounding), and ||H| - 1| <= 2e-4 J at distance >=
    delta/2 from every band (each notch's pass-band ripple adds up)."""
    _, taps, _ = design(fs, centers, widths, ntaps)
    d = delta(fs, taps.size)
    M = 1 << 19
    mag = np.abs(np.fft.fft(taps.astype(np.complex128), M))
    f = np.fft.fftfreq(M, 1.0 / fs)
    core, far = np.zeros(M, bool), np.ones(M, bool)
    for c, w in zip(centers, widths):
        core |= (f >= c - w / 2 + d / 2) & (f <= c + w / 2 - d / 2)
        for sh in (-fs, 0, fs):
            far &= np.maximum(np.maximum(c + sh - w / 2 - f, f - (c + sh + w / 2)), 0.0) >= d / 2
    assert core.any() and far.any()
    assert mag[core].max() <= 2e-4
    assert np.abs(mag[far] - 1.0).max() <= 2e-4 * len(centers)


def test_default_ntaps_and_fft_size_rules():
    # L = the smallest odd value >= 65 with w_min >= 2 delta(L); N = the smallest power of two >= 2 (L - 1), at least 1024
    for fs, widths in [(10_000_000, [200e3, 100e3]), (2_000_000, [10e3]), (8_000_000, [1e6]), (100_000_000, [1e6, 3e6]),
                       (20_000_000, [24_600.0]), (48_000, [2_000.0])]:
        _, taps, nfft = design(fs, [0.0] + [fs / 4] * (len(widths) - 1), widths)
        L = taps.size
        wmin = min(widths)
        assert L % 2 == 1 and L >= 65 and wmin >= 2 * delta(fs, L)
        assert L == 65 or wmin < 2 * delta(fs, L - 2), (fs, widths, L)
        assert nfft == max(1024, 1 << int(np.ceil(np.log2(2 * (L - 1))))) and nfft <= 16384
    for L, N in [(65, 1024), (513, 1024), (515, 2048), (1025, 2048), (4097, 8192), (8193, 16384)]:
        assert design(8_000_000, [0.0], [2e6], L)[2] == N


@pytest.mark.parametrize("cfg,text", [
    ((8_000_000, [], [], 0), "the number of notches must be in 1..32"),
    ((8_000_000, list(np.arange(33) * 1e5 - 3e6), [2e4] * 33, 0), "the number of notches must be in 1..32"),
    ((8_000_000, [0.0], [0.0], 0), "every width must be > 0"),
    ((8_000_000, [0.0], [-1e5], 0), "every width must be > 0"),
    ((8_000_000, [float("nan")], [1e5], 0), "every center must be finite"),
    ((8_000_000, [3.96e6], [1e5], 0), "inside the capture (|center| + width / 2 <= fs / 2)"),
    ((8_000_000, [-4e6], [1e5], 0), "inside the capture (|center| + width / 2 <= fs / 2)"),
    ((8_000_000, [0.0], [1e5], 64), "ntaps must be odd, in 65..8193"),
    ((8_000_000, [0.0], [1e5], 63), "ntaps must be odd, in 65..8193"),
    ((8_000_000, [0.0], [1e5], 8195), "ntaps must be odd, in 65..8193"),
    ((8_000_000, [0.0], [1e5], 65), "at least twice the transition width"),
    ((8_000_000, [0.0], [9e3], 0), "needs more than 8193 taps"),
    ((8_000_000, [0.0, 1.5e5], [2e5, 1e5], 0), "merge them into one"),
    ((8_000_000, [0.0, 1e5], [2e5, 2e5], 0), "merge them into one"),
    ((8_000_000, [-3.9e6, 3.9e6], [2e5, 2e5], 0), "merge them into one"),          # neighbours across +-fs/2
])
def test_invalid_configurations_are_rejected_with_their_rule(cfg, text):
    lib = _native.lib()
    fs, c, w, L = cfg
    ca, wa = np.ascontiguousarray(c, np.float64), np.ascontiguousarray(w, np.float64)
    assert lib.tsdrgpu_notch_design(fs, ca.size, ca.ctypes.data_as(C.c_void_p), wa.ctypes.data_as(C.c_void_p), L, None, 0, None, None) == -3
    assert text in lib.tsdrgpu_last_error(None).decode()
    # the edges are allowed: a band touching +-fs/2, two bands exactly delta(L) apart, a width of exactly 2 delta(L)
    d = delta(8_000_000, 1025)
    for c, w in [([3.9e6], [2e5]), ([0.0, 3 * d], [2 * d, 2 * d]), ([0.0], [2 * d])]:
        assert design(8_000_000, c, w, 1025)[0] == 0, (c, w)


@pytest.mark.parametrize("nfft,ok", [(64, True), (16384, True), (4096, True), (32, False), (32768, False), (100, False), (0, False)])
def test_spectrum_rules(nfft, ok):
    lib = _native.lib()
    assert (lib.tsdrgpu_spectrum_check(8_000_000, nfft) == 0) == ok
    if not ok:
        assert "nfft must be a power of two in 64..16384" in lib.tsdrgpu_last_error(None).decode()


def test_host_library_rejects_malformed_notch_and_spectrum_knobs(tmp_path, monkeypatch):
    """TSDR_NOTCH, TSDR_NOTCH_TAPS and TSDR_SPECTRUM are checked before any device work: a malformed or invalid value fails
    tsdr_readasync with TSDR_INVALID_PARAMETER_VALUE and a text naming what is wrong."""
    from tempestsdr_b200 import synth
    from tests.test_host_library import FRAME_CB, MINE, PLOT_CB, PLUGIN, VALUE_CB, bind
    raw = tmp_path / "iq.raw"
    synth.noise_iq(4096, seed=1).tofile(raw)
    lib = bind(MINE)
    t = C.c_void_p()
    nv, npl = VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
    lib.tsdr_init(C.byref(t), nv, npl, None)
    lib.tsdr_setresolution(t, 125, 60.0)
    assert lib.tsdr_loadplugin(t, PLUGIN.encode(), f'"{raw}" 8000000 float'.encode()) == 0
    cases = [({"TSDR_NOTCH": "abc"}, b"TSDR_NOTCH: expected"), ({"TSDR_NOTCH": "1e6"}, b"TSDR_NOTCH: expected"),
             ({"TSDR_NOTCH": "1e6:2e5,"}, b"TSDR_NOTCH: expected"), ({"TSDR_NOTCH": "1e6:2e5;3e5:1e5"}, b"TSDR_NOTCH: expected"),
             ({"TSDR_NOTCH": "1e6:"}, b"TSDR_NOTCH: expected"),
             ({"TSDR_NOTCH": ",".join(f"{k * 1e5}:2e4" for k in range(33))}, b"TSDR_NOTCH: at most 32 notches"),
             ({"TSDR_NOTCH": "3.95e6:2e5"}, b"|center| + width / 2 <= fs / 2"),
             ({"TSDR_NOTCH": "0:2e5,1.5e5:1e5"}, b"merge them into one"),
             ({"TSDR_NOTCH": "0:2e5", "TSDR_NOTCH_TAPS": "x"}, b"TSDR_NOTCH_TAPS: expected"),
             ({"TSDR_NOTCH": "0:2e5", "TSDR_NOTCH_TAPS": "64"}, b"ntaps must be odd, in 65..8193"),
             ({"TSDR_SPECTRUM": "4096x", "TSDR_SPECTRUM_FILE": str(tmp_path / "s.csv")}, b"TSDR_SPECTRUM: expected"),
             ({"TSDR_SPECTRUM": "1000", "TSDR_SPECTRUM_FILE": str(tmp_path / "s.csv")}, b"power of two in 64..16384"),
             ({"TSDR_SPECTRUM": "4096"}, b"TSDR_SPECTRUM: needs TSDR_SPECTRUM_FILE")]
    for env, text in cases:
        for k in ("TSDR_NOTCH", "TSDR_NOTCH_TAPS", "TSDR_SPECTRUM", "TSDR_SPECTRUM_FILE"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        assert lib.tsdr_readasync(t, FRAME_CB(lambda *a: None), None) == 9, env        # TSDR_INVALID_PARAMETER_VALUE
        assert text in lib.tsdr_getlasterrortext(t), env
        assert lib.tsdr_isrunning(t) == 0
    lib.tsdr_free(C.byref(t))


# ---------------------------------------------------------------------------------------------------------------- GPU helpers

def assemble(segments):
    """x~ over the whole stream (zeros over every drop) and each block's span.  segments: [(dropped_before, complex block)]."""
    total = sum(g + b.size for g, b in segments)
    x = np.zeros(total, np.complex128)
    spans, pos = [], 0
    for g, b in segments:
        pos += g
        x[pos:pos + b.size] = b
        spans.append((pos, b.size))
        pos += b.size
    return x, spans


def notch_model(segments, taps):
    x, spans = assemble(segments)
    y = scipy.signal.oaconvolve(x, taps.astype(np.complex128))[: x.size]
    return [y[b0:b0 + k] for b0, k in spans]


def welch_model(segments, fs, nfft):
    """Welch over the complete segments at multiples of nfft/2 that touch no dropped position, fft-shifted."""
    x, spans = assemble(segments)
    valid = np.zeros(x.size, bool)
    for b0, k in spans:
        valid[b0:b0 + k] = True
    w = scipy.signal.get_window("hann", nfft)
    acc, n = np.zeros(nfft), 0
    for s in range(0, (x.size - nfft) // (nfft // 2) + 1 if x.size >= nfft else 0):
        a = s * nfft // 2
        if valid[a:a + nfft].all():
            acc += np.abs(np.fft.fft(x[a:a + nfft] * w)) ** 2
            n += 1
    return np.fft.fftshift(acc / (n * fs * np.sum(w ** 2))) if n else np.zeros(nfft), n


def tones(n, fs, freqs, amps, seed, noise=0.3):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    z = noise * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    for f, a in zip(freqs, amps):
        z = z + a * np.exp(2j * np.pi * f / fs * t + 1j * rng.uniform(0, 6.28))
    return z


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("fs,centers,widths,ntaps,fmt", [
    (10_000_000, [1e6, -2e6], [200e3, 100e3], 0, "float32"),
    (8_000_000, [-3.85e6, 0.0, 1.5e6], [100e3, 40e3, 300e3], 0, "int8"),
    (100_000_000, list(np.linspace(-40e6, 40e6, 32)), [1e6] * 32, 0, "float32"),
    (25_000_000, [1e6, 1.3e6, 1.6e6], [100e3, 100e3, 100e3], 8193, "float32"),
    (8_000_000, [2e6], [1.4e6], 65, "float32"),
    (8_000_000, [-1e6, 2.5e6], [5e5, 5e5], 4097, "int8"),
])
def test_stage_matches_float64_model(fs, centers, widths, ntaps, fmt):
    import torch
    from tempestsdr_b200 import api
    ctx = api.Context(0)
    nt = ctx.notch()
    nt.configure(fs, centers, widths, ntaps)
    taps = nt.taps()
    L = taps.size
    z = tones(300_000, fs, [centers[0], centers[-1] + widths[-1], 0.123 * fs], [3.0, 1.0, 0.5], seed=L)
    # sizes cover a block shorter than the history, empty blocks, a loss-only block and drops of several lengths
    sizes = [0, 1, 17, 70_000, 3, 0, L // 3, 100_000, 29_000, 101_000]
    drops = [0, 0, 5, 0, 1234, 777, 0, L + 1, 3, 0]
    segs, got, gotd, o = [], [], [], 0
    for k, g in zip(sizes, drops):
        blk = z[o:o + k]; o += k
        if fmt == "int8":
            q = np.clip(np.round(iq(blk) * 20.0), -128, 127).astype(np.int8)
            x = ctx.convert_samples(torch.from_numpy(q).cuda())
            blk = cplx((q.astype(np.float64) / 128.0).astype(np.float32))
        else:
            x = torch.from_numpy(iq(blk)).cuda()
        segs.append((g, blk))
        out, od = nt.run(x, g)
        got.append(out.cpu().numpy()); gotd.append(od)
    want = notch_model(segs, taps)
    peak = max(np.max(np.abs(b)) for _, b in segs if b.size)
    worst = 0.0
    for k, (g_, w) in enumerate(zip(got, want)):
        assert g_.size == 2 * w.size, k
        if w.size:
            worst = max(worst, float(np.max(np.abs(cplx(g_) - w))))
    assert gotd == drops
    print(f"L={L} J={len(centers)} {fmt}: max error / input peak = {worst / peak:.2e}")
    assert worst <= 1e-5 * peak


def _run_cut(nt, x_all, bounds, drops_at):
    import torch
    outs, pending = [], dict(drops_at)
    for a, b in zip(bounds[:-1], bounds[1:]):
        out, od = nt.run(torch.from_numpy(x_all[2 * a:2 * b].copy()).cuda(), pending.pop(a, 0))
        outs.append(out.cpu().numpy())
    assert not pending
    return np.concatenate(outs)


@pytest.mark.gpu
@pytest.mark.parametrize("ntaps", [65, 1025, 8193])
def test_block_cuts(ntaps):
    """Cuts at multiples of the hop (also through drops that keep the cut points there) give bit-identical outputs; arbitrary cuts
    agree to 2e-6 of the peak (FFT round-off of the partial segments)."""
    from tempestsdr_b200 import api
    fs = 24_000_000
    ctx = api.Context(0)
    z = tones(400_000, fs, [2e6, -5e6], [1.0, 2.0], seed=ntaps)
    x_all = iq(z)
    nt = ctx.notch()
    nt.configure(fs, [2e6], [4e6], ntaps)
    hop = nt.nfft - (ntaps - 1)
    rng = np.random.default_rng(ntaps)
    drops_at = {3 * hop: 2 * hop, 9 * hop: hop}                  # data index -> lost pairs before it (multiples of the hop)
    aligned = []
    for cut in range(2):
        nt.reset()
        b, bounds = 0, [0]
        while b < z.size:
            b = min(b + hop * int(rng.integers(1, 6)), z.size) if cut else min(b + hop, z.size)
            bounds.append(b)
        for d in drops_at:
            if d not in bounds:
                bounds = sorted(bounds + [d])
        aligned.append(_run_cut(nt, x_all, bounds, drops_at))
    assert np.array_equal(aligned[0].view(np.uint32), aligned[1].view(np.uint32))
    nt.reset()
    b, bounds = 0, [0]
    while b < z.size:
        b = min(b + int(rng.choice([1, 7, ntaps - 2, int(rng.integers(1, 30_000))])), z.size)
        bounds.append(b)
    bounds = sorted(set(bounds) | set(drops_at))
    rnd = _run_cut(nt, x_all, bounds, drops_at)
    peak = np.max(np.abs(z))
    err = np.max(np.abs(cplx(rnd) - cplx(aligned[0])))
    print(f"L={ntaps}: random cuts differ by {err / peak:.2e} of the peak")
    assert err <= 2e-6 * peak


@pytest.mark.gpu
@pytest.mark.parametrize("fs,centers,widths", [(8_000_000, [-1.2e6, 0.3e6, 1.7e6], [200e3, 100e3, 300e3]),
                                               (100_000_000, [-11e6, 4e6], [2e6, 1e6])])
def test_in_band_tones_are_removed(fs, centers, widths):
    """notch(raster + tones at the notches' centres, each 10x the raster) - notch(raster) stays below 3e-4 of the tone
    amplitude past the first L pairs."""
    import torch
    from tempestsdr_b200 import api
    ctx = api.Context(0)
    n = 400_000
    r, _ = emitter(n, fs, 60.0, 125, 3, 1.0, 0.0, fs // 4)
    r = r / np.max(np.abs(r))
    amp = 10.0
    t = np.arange(n)
    tone = sum(amp * np.exp(2j * np.pi * (c + 0.1 * w) / fs * t + 1j * k) for k, (c, w) in enumerate(zip(centers, widths)))
    nt = ctx.notch()
    nt.configure(fs, centers, widths)
    L = nt.taps().size
    outs = []
    for sig in (r + tone, r):
        nt.reset()
        outs.append(cplx(nt.run(torch.from_numpy(iq(sig)).cuda())[0].cpu().numpy()))
    diff = np.max(np.abs(outs[0][L:] - outs[1][L:]))
    print(f"residual of the tones: {diff / amp:.2e} of their amplitude")
    assert diff <= 3e-4 * amp


@pytest.mark.gpu
@pytest.mark.parametrize("nfft", [64, 256, 1024, 4096, 16384])
def test_spectrum_matches_welch(nfft):
    import torch
    from tempestsdr_b200 import api
    fs = 20_000_000
    ctx = api.Context(0)
    z = tones(200_003, fs, [1e6, -7.3e6, 3.3e6], [5.0, 1.0, 0.01], seed=nfft)
    sp = ctx.spectrum()
    sp.configure(fs, nfft)
    sp.run(torch.from_numpy(iq(z)).cuda())
    f, psd, segs = sp.result()
    wf, wp = scipy.signal.welch(z, fs, window="hann", nperseg=nfft, noverlap=nfft // 2, detrend=False, return_onesided=False,
                                scaling="density")
    wp, wf = np.fft.fftshift(wp), np.fft.fftshift(wf)
    assert segs == (z.size - nfft) // (nfft // 2) + 1
    assert np.array_equal(f, wf) or np.max(np.abs(f - wf)) <= 1e-6 * fs
    err = np.max(np.abs(psd - wp)) / np.max(wp)
    print(f"nfft={nfft}: max error / peak bin = {err:.2e}")
    assert err <= 1e-5


@pytest.mark.gpu
def test_spectrum_skips_segments_with_drops_and_ignores_the_cut():
    import torch
    from tempestsdr_b200 import api
    fs, nfft = 10_000_000, 1024
    ctx = api.Context(0)
    z = tones(300_000, fs, [1e6, -3e6], [2.0, 1.0], seed=11)
    sizes = [0, 5000, 3, 0, 70_000, 511, 100_000, 124_486]
    drops = [0, 0, 700, 10, 0, 1, 5000, 0]
    results = []
    for cut in range(3):
        sp = ctx.spectrum()
        sp.configure(fs, nfft)
        rng = np.random.default_rng(cut)
        o, segs = 0, []
        for k, g in zip(sizes, drops):
            blk = z[o:o + k]; o += k
            segs.append((g, blk))
            parts = np.sort(rng.integers(0, k + 1, size=3 * cut)) if cut else np.array([], int)
            edges = [0] + list(parts) + [k]
            for i, (a, b) in enumerate(zip(edges[:-1], edges[1:])):        # the drop goes with the first piece
                sp.run(torch.from_numpy(iq(blk[a:b])).cuda(), g if i == 0 else 0)
        results.append(sp.result())
    want, n = welch_model(segs, fs, nfft)
    assert n > 0 and results[0][2] == n
    assert np.max(np.abs(results[0][1] - want)) <= 1e-5 * np.max(want)
    for r in results[1:]:
        assert r[2] == n and np.array_equal(r[1].view(np.uint64), results[0][1].view(np.uint64))


def _feed(p, blk, d, fmt):
    if fmt == "int8":
        p.process_raw(blk, d)
    else:
        p.process(blk, d)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,tuned", [("float32", False), ("int8", False), ("float32", True), ("int8", True)])
def test_pipeline_is_the_notch_then_the_unnotched_pipeline(fmt, tuned):
    """A notched pipeline delivers exactly what an un-notched pipeline delivers when fed, block by block, the stage notch's
    output: frames, plots and values bit-identical, with drops and a loss-only block in the stream.  A spectrum set on the
    notched pipeline changes none of it and equals the stage spectrum of the blocks as received."""
    import torch
    from tempestsdr_b200 import api, synth
    fs, h, fv, items, nblk = 8_000_000, 125, 60.0, 65536, 44
    centers, widths = [-2.2e6, 0.7e6, 3.1e6], [200e3, 100e3, 300e3]
    w = int(2 * fs / (fv * h))
    z = cplx(synth.video_like_iq(nblk * items // 2, fs, w, h, fv, seed=21))
    t = np.arange(z.size)
    z = z + sum(0.8 * np.exp(2j * np.pi * c / fs * t) for c in centers)
    if fmt == "int8":
        data = np.clip(np.round(iq(z) * 40.0), -128, 127).astype(np.int8)
        as_float = lambda b: (b.astype(np.float64) / 128.0).astype(np.float32)
    else:
        data = iq(z)
        as_float = lambda b: b
    drops = {3: 3, 5: 40_001, 6: 1, 40: 123_457, 42: 2 * items}
    p1, g1 = _collect_pipeline(fs, h, fv)
    p1.set_notches(centers, widths)
    p1.set_spectrum(2048)
    p2, g2 = _collect_pipeline(fs, h, fv)
    if tuned:
        p1.set_tuner(1e6, 2e6, 4)
        p2.set_tuner(1e6, 2e6, 4)
    ctx = api.Context(0)
    nt = ctx.notch()
    nt.configure(fs, centers, widths)
    sp = ctx.spectrum()
    sp.configure(fs, 2048)
    for k in range(nblk):
        blk = data[k * items:(k + 1) * items].copy()
        d = drops.get(k, 0)
        if k == 41:                                                  # an empty block that only reports a loss
            p1.process(np.zeros(0, np.float32), 999)
            out, od = nt.run(torch.zeros(0, dtype=torch.float32, device="cuda"), 999)
            sp.run(torch.zeros(0, dtype=torch.float32, device="cuda"), 999)
            p2.process(out.cpu().numpy(), od)
        _feed(p1, blk, d, fmt)
        x = torch.from_numpy(as_float(blk)).cuda()
        sp.run(x, d)
        out, od = nt.run(x, d)
        p2.process(out.cpu().numpy(), od)
    p1.flush(); p2.flush()
    assert len(g1["frames"]) >= 3 and len(g1["plots"]) >= 2
    _same(g1, g2)
    f1, psd1, n1 = p1.spectrum()
    f2, psd2, n2 = sp.result()
    assert n1 == n2 > 0 and np.array_equal(f1, f2) and np.array_equal(psd1.view(np.uint64), psd2.view(np.uint64))
    p1.close(); p2.close()


@pytest.mark.gpu
def test_spectrum_leaves_the_pipeline_unchanged():
    from tempestsdr_b200 import synth
    fs, h, fv, items = 8_000_000, 125, 60.0, 65536
    x = synth.video_like_iq(30 * items // 2, fs, int(2 * fs / (fv * h)), h, fv, seed=5)
    runs = []
    for nfft in (0, 4096):
        p, g = _collect_pipeline(fs, h, fv)
        p.set_spectrum(nfft)
        for k in range(30):
            p.process(x[k * items:(k + 1) * items].copy(), 7 if k == 9 else 0)
        p.flush()
        runs.append((g, p.spectrum()))
        p.close()
    _same(runs[0][0], runs[1][0])
    assert runs[0][1][1].size == 0 and runs[1][1][2] > 0


def carriers_case(fs=8_000_000, secs=0.5, seed=5):
    """One emitter at 0 Hz, 2 MHz wide, and three carriers inside its band, each 3x its peak magnitude."""
    n = int(fs * secs)
    e, raster = emitter(n, fs, 60.0, 125, seed, 1.0, 0.0, 2_000_000)
    peak = np.max(np.abs(e))
    rng = np.random.default_rng(seed + 2)
    t = np.arange(n)
    freqs = [-0.61e6, 0.23e6, 0.77e6]
    z = e + sum(3.0 * peak * np.exp(2j * np.pi * f / fs * t + 1j * rng.uniform(0, 6.28)) for f in freqs)
    z = z + 0.02 * peak * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return iq(z), raster, freqs


# raster_corr's scale: 0.56 for a perfect copy.  Through the oracle (test_carriers_case_through_the_oracle: float64 notch and
# tuner, then the oracle's demod, resampler and frame stage) the last four frames correlate at 0.009 without the notches and at
# 0.467, at one alignment, with 60 kHz stopbands around the carriers.  The thresholds: un-notched below CARRIERS_MAX, notched at
# OWN_MIN (0.3) or more at one alignment.
CARRIERS_MAX = 0.15
NOTCH_WIDTH = 60e3


def test_carriers_case_through_the_oracle():
    from oracle import oracle as orc
    from tempestsdr_b200 import api
    O = orc.best()
    fs, D, h, fv = 8_000_000, 4, 125, 60.0
    x, raster, freqs = carriers_case(fs)
    z = cplx(x)
    taps_t, _ = api.tuner_design(fs, 0.0, 2_000_000, D)
    res = {}
    for notched in (False, True):
        y = z
        if notched:
            tn, _ = api.notch_design(fs, freqs, [NOTCH_WIDTH] * 3)
            y = scipy.signal.oaconvolve(z, tn.astype(np.complex128))[: z.size]
        u = scipy.signal.oaconvolve(y, taps_t.astype(np.float64))[: y.size][::D]
        fsi = fs // D
        w, _, _ = O.geometry(fsi, h, fv)
        mag = O.am_demod(iq(u))
        rs = O.resampler()
        blk = int(0.1 * fsi / fv)
        pix = np.concatenate([rs.run(mag[k * blk:(k + 1) * blk], w * h * fv, fsi) for k in range(mag.size // blk)])
        n = w * h
        po = O.postprocessor(fsi, h, fv, 1, 0)
        frames = [po.run(pix[k * n:(k + 1) * n], w, h, 0.0, 0.1, 1, 0)[0].copy() for k in range(pix.size // n)]
        res[notched] = [raster_corr(f, w, raster) for f in frames[-4:]]
    print(f"oracle: un-notched {res[False]}, notched {res[True]}")
    assert max(c for c, _ in res[False]) < CARRIERS_MAX
    assert min(c for c, _ in res[True]) >= OWN_MIN and len({i for _, i in res[True]}) == 1


@pytest.mark.gpu
def test_notches_recover_the_picture_the_carriers_hide():
    fs = 8_000_000
    x, raster, freqs = carriers_case(fs)
    items = 65536
    pn, gn = _collect_pipeline(fs, 125, 60.0)
    pu, gu = _collect_pipeline(fs, 125, 60.0)
    pn.set_notches(freqs, [NOTCH_WIDTH] * 3)
    pn.set_tuner(0, 2_000_000, 4)
    pu.set_tuner(0, 2_000_000, 4)
    for k in range(x.size // items):
        blk = x[k * items:(k + 1) * items].copy()
        pn.process(blk, 0); pu.process(blk, 0)
    pn.flush(); pu.flush()
    assert len(gn["frames"]) >= 8 and len(gu["frames"]) >= 8
    cn = [raster_corr(f, w, raster) for w, f in gn["frames"][-4:]]
    cu = [raster_corr(f, w, raster)[0] for w, f in gu["frames"][-4:]]
    print(f"carriers: notched {cn}, un-notched {cu}")
    assert min(c for c, _ in cn) >= OWN_MIN and len({i for _, i in cn}) == 1, cn
    assert max(cu) < CARRIERS_MAX, cu
    pn.close(); pu.close()


@pytest.mark.gpu
def test_live_reconfiguration_and_switching_off():
    """Changing the notches mid-run works without an error; switching them off gives frames bit-identical to a never-notched
    pipeline fed the rest of the stream."""
    from tempestsdr_b200 import synth
    fs, h, fv, items = 8_000_000, 125, 60.0, 65536
    x = synth.video_like_iq(60 * items // 2, fs, int(2 * fs / (fv * h)), h, fv, seed=9)
    p, g = _collect_pipeline(fs, h, fv)
    p.set_notches([1e6], [2e5])
    for k in range(20):
        p.process(x[k * items:(k + 1) * items].copy(), 0)
    p.set_notches([-1e6, 2e6], [1e5, 3e5], 2049)
    p.process(x[20 * items:21 * items].copy(), 0)
    n_before = len(g["frames"])
    p.set_notches([], [])                                 # off
    for k in range(21, 60):
        p.process(x[k * items:(k + 1) * items].copy(), 0)
    p.flush()
    q, gq = _collect_pipeline(fs, h, fv)
    for k in range(21, 60):
        q.process(x[k * items:(k + 1) * items].copy(), 0)
    q.flush()
    after = g["frames"][n_before:]
    assert len(after) == len(gq["frames"]) >= 3
    for (wa, fa), (wb, fb) in zip(after, gq["frames"]):
        assert wa == wb and np.array_equal(fa.view(np.uint32), fb.view(np.uint32))
    with pytest.raises(_native.TsdrGpuError, match="merge them into one"):
        p.set_notches([0.0, 1e5], [2e5, 2e5])
    with pytest.raises(_native.TsdrGpuError, match=r"\|center\| \+ width / 2 <= fs / 2"):
        p.set_notches([3.5e6], [2e5])
        p.set_samplerate(4_000_000)
    p.close(); q.close()


@pytest.mark.gpu
def test_superbandwidth_mode_bypasses_and_resumes_both_stages():
    from tempestsdr_b200 import synth
    fs, h, fv = 400_000, 80, 50.0
    items = 16384
    nblk = 2 * (4 * (10 * int(fs / fv) + int(0.5 * fs)) // (items // 2) + 8)
    x = synth.video_like_iq(nblk * items // 2, fs, 200, 80, fv, seed=41, snr_db=25)
    outs = []
    for staged in (False, True):
        p, g = _collect_pipeline(fs, h, fv, on_retune=lambda off: None)
        if staged:
            p.set_notches([50_000], [20_000])
            p.set_spectrum(1024)
        p.set_param("superresolution", 1)
        for k in range(nblk):
            p.process(x[k * items:(k + 1) * items].copy(), 0)
        p.flush()
        spec = p.spectrum()
        outs.append(({"frames": list(g["frames"])}, spec))
        if staged:                                        # the mode ends: both stages resume, reset
            p.set_param("superresolution", 0)
            for k in range(8):
                p.process(x[k * items:(k + 1) * items].copy(), 0)
            p.flush()
            f, psd, segs = p.spectrum()
            assert segs == (8 * items // 2 - 1024) // 512 + 1
        p.close()
    assert len(outs[0][0]["frames"]) >= 4
    assert [w for w, _ in outs[0][0]["frames"]] == [w for w, _ in outs[1][0]["frames"]]
    for (_, a), (_, b) in zip(outs[0][0]["frames"], outs[1][0]["frames"]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert outs[1][1][2] == 0                             # nothing reached the spectrum while the mode ran


@pytest.mark.gpu
def test_host_library_notch_and_spectrum_knobs(tmp_path, monkeypatch):
    from tests.test_host_library import FRAME_CB, MINE, PLOT_CB, PLUGIN, VALUE_CB, bind
    fs, D = 8_000_000, 4
    x, raster, freqs = carriers_case(fs, secs=0.4)
    raw = tmp_path / "carriers.raw"
    x.tofile(raw)
    csv = tmp_path / "spectrum.csv"
    got = []
    monkeypatch.setenv("TSDR_NO_DROP", "1")
    monkeypatch.setenv("TSDR_NO_RAW_SINK", "1")
    monkeypatch.setenv("TSDR_TUNER", "0,2000000,4")
    monkeypatch.setenv("TSDR_NOTCH", ",".join(f"{f}:{NOTCH_WIDTH}" for f in freqs))
    monkeypatch.setenv("TSDR_SPECTRUM", "4096")
    monkeypatch.setenv("TSDR_SPECTRUM_FILE", str(csv))
    lib = bind(MINE)
    t = C.c_void_p()
    nv, npl = VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
    fcb = FRAME_CB(lambda b, ww, hh, c: got.append((ww, np.ctypeslib.as_array(b, shape=(ww * hh,)).copy())))
    lib.tsdr_init(C.byref(t), nv, npl, None)
    lib.tsdr_setresolution(t, 125, 60.0); lib.tsdr_motionblur(t, 0.0); lib.tsdr_setgain(t, 0.5)
    for pid, v in ((0, 1), (1, 0), (6, 1)):
        lib.tsdr_setparameter_int(t, pid, v)
    assert lib.tsdr_loadplugin(t, PLUGIN.encode(), f'"{raw}" {fs} float'.encode()) == 0
    rc = []
    th = threading.Thread(target=lambda: rc.append(lib.tsdr_readasync(t, fcb, None)))
    th.start()
    deadline = time.time() + 60
    while len(got) < 12 and time.time() < deadline:
        time.sleep(0.05)
    assert lib.tsdr_stop(t) == 0
    th.join(timeout=30)
    assert rc == [0]
    assert len(got) >= 12 and all(w == int(2 * (fs // D) / (60.0 * 125)) for w, _ in got)
    c = [raster_corr(f, w, raster)[0] for w, f in got[8:12]]
    assert min(c) >= OWN_MIN, c
    lib.tsdr_free(C.byref(t))
    rows = np.loadtxt(csv, delimiter=",", skiprows=1)
    assert rows.shape == (4096, 2) and np.all(np.diff(rows[:, 0]) > 0)
    assert rows[0, 0] == -fs / 2 and rows[-1, 0] == fs / 2 - fs / 4096
    top = rows[np.argsort(rows[:, 1])[-3:], 0]
    for f in freqs:                                       # the three carriers are the three highest bins
        assert np.min(np.abs(top - f)) <= fs / 4096, (f, top)
