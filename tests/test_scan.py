"""The channelizer (polyphase filter bank, csrc/channelizer.cu) and the scan built on it (a frame-rate detector per channel): the
prototype against firwin and the tuner's design, the configuration rules, the kernel against a float64 model and against the tuner
channel by channel, block-cut invariance, the scan against a float64 model of the whole scan, the two-emitter use case (scan, then
tune), the pipeline's scan beside an untouched pixel path, and the host library's TSDR_SCAN knob."""
import ctypes as C
import os
import threading
import time

import numpy as np
import pytest
import scipy.signal

from tempestsdr_b200 import _native
from tests.test_tuner import BETA, OWN_MIN, _collect_pipeline, _same, cplx, design, emitter, iq, raster_corr, tone_signal


def ch_design(fs, K, Q=0):
    lib = _native.lib()
    taps = np.zeros(8192, np.float32)
    n = C.c_int(0)
    rc = lib.tsdrgpu_channelizer_design(fs, K, Q, taps.ctypes.data_as(C.c_void_p), taps.size, C.byref(n))
    return rc, taps[: n.value]


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("fs,K,Q", [(8_000_000, 2, 4), (8_000_000, 8, 16), (32_000_000, 8, 0), (64_000_000, 64, 16),
                                    (100_000_000, 64, 32), (200_000_000, 256, 16), (34_000_000, 256, 32), (2_000_000, 4, 8)])
def test_design_matches_firwin_and_the_tuner(fs, K, Q):
    rc, taps = ch_design(fs, K, Q)
    assert rc == 0
    n = (Q or 16) * K - 1
    want = scipy.signal.firwin(n, fs / (2 * K), window=("kaiser", BETA), fs=fs)
    assert taps.size == n and np.max(np.abs(taps.astype(np.float64) - want)) <= 1e-7
    if K // 2 <= 64 and n <= 1023:                             # the tuner's own limits
        rc, tt, _ = design(fs, 0.0, fs / K, K // 2, n)
        assert rc == 0 and np.array_equal(tt.view(np.uint32), taps.view(np.uint32))


@pytest.mark.parametrize("cfg,text", [
    ((8_000_000, 3, 16), "channels must be a power of two in 2..256"),
    ((8_000_000, 1, 16), "channels must be a power of two in 2..256"),
    ((8_000_000, 512, 16), "channels must be a power of two in 2..256"),
    ((8_000_000, 0, 16), "channels must be a power of two in 2..256"),
    ((8_000_000, 8, 3), "taps_per_channel must be in 4..32 (0 = default)"),
    ((8_000_000, 8, 33), "taps_per_channel must be in 4..32 (0 = default)"),
    ((8_000_002, 8, 16), "multiple of channels / 2 (fs % (K/2) == 0)"),
    ((8_000_000, 128, 16), "channel rate 2 fs / K must be at least 130500"),
    ((520_000, 8, 16), "channel rate 2 fs / K must be at least 130500"),
])
def test_invalid_configurations_are_rejected_with_their_rule(cfg, text):
    lib = _native.lib()
    assert lib.tsdrgpu_channelizer_design(*cfg, None, 0, None) == -3          # TSDRGPU_EINVAL
    assert text in lib.tsdrgpu_last_error(None).decode()
    # the edges are allowed; the shared-memory rule holds for every K and Q the other rules let through (largest tile: K = 256, Q = 32)
    assert lib.tsdrgpu_channelizer_design(522_000, 8, 16, None, 0, None) == 0
    assert lib.tsdrgpu_channelizer_design(2 ** 24, 256, 32, None, 0, None) == 0


def test_out_pairs_is_the_tuners_arithmetic_at_half_the_channels():
    lib = _native.lib()
    rng = np.random.default_rng(3)
    a, ad, b, bd = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    for _ in range(2000):
        K = int(rng.choice([2, 4, 8, 64, 128]))
        pos, k, g = (int(v) for v in rng.integers(0, 10 ** 7, 3))
        assert lib.tsdrgpu_channelizer_out_pairs(pos, k, g, K, C.byref(a), C.byref(ad)) == 0
        assert lib.tsdrgpu_tuner_out_pairs(pos, k, g, K // 2, C.byref(b), C.byref(bd)) == 0
        assert (a.value, ad.value) == (b.value, bd.value)
    assert lib.tsdrgpu_channelizer_out_pairs(0, 1000, 0, 256, C.byref(a), C.byref(ad)) == 0 and a.value == 8
    assert lib.tsdrgpu_channelizer_out_pairs(0, 1, 0, 6, C.byref(a), C.byref(ad)) == -3


def test_host_library_rejects_a_malformed_scan_knob(tmp_path, monkeypatch):
    """TSDR_SCAN is checked before any device work: a malformed or invalid value, or TSDR_SCAN without TSDR_SCAN_FILE, fails
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
    monkeypatch.setenv("TSDR_SCAN_FILE", str(tmp_path / "scan.csv"))
    for value, text in [("abc", b"TSDR_SCAN: expected"), ("8,", b"TSDR_SCAN: expected"), ("8,16,2", b"TSDR_SCAN: expected"),
                        ("8.5", b"TSDR_SCAN: expected"), ("-8", b"TSDR_SCAN: expected"), ("6", b"power of two in 2..256"),
                        ("8,40", b"taps_per_channel must be in 4..32"), ("128", b"at least 130500")]:
        monkeypatch.setenv("TSDR_SCAN", value)
        assert lib.tsdr_readasync(t, FRAME_CB(lambda *a: None), None) == 9, value        # TSDR_INVALID_PARAMETER_VALUE
        assert text in lib.tsdr_getlasterrortext(t), value
        assert lib.tsdr_isrunning(t) == 0
    monkeypatch.delenv("TSDR_SCAN_FILE")
    monkeypatch.setenv("TSDR_SCAN", "8")
    assert lib.tsdr_readasync(t, FRAME_CB(lambda *a: None), None) == 9
    assert b"TSDR_SCAN_FILE" in lib.tsdr_getlasterrortext(t)
    lib.tsdr_free(C.byref(t))


# ---------------------------------------------------------------------------------------------------------------- models

def offsets(fs, K):
    c = np.arange(K)
    return np.where(c < K // 2, c, c - K) * (fs / K)


def channelizer_model(segments, taps, K):
    """float64 model: zero-fill every gap, mix channel c by e^{-2 pi i c n / K} (exact phase), filter, keep every (K/2)-th output
    inside a block.  segments: [(dropped_before, complex block)].  Returns, per block, a [K, M] complex array."""
    D = K // 2
    total = sum(g + b.size for g, b in segments)
    x = np.zeros(total, np.complex128)
    spans, pos = [], 0
    for g, b in segments:
        pos += g
        x[pos:pos + b.size] = b
        spans.append((pos, b.size))
        pos += b.size
    n = np.arange(total, dtype=np.int64)
    ms = [np.arange(-(-b0 // D), -(-(b0 + k) // D), dtype=np.int64) * D for b0, k in spans]
    out = [np.zeros((K, m.size), np.complex128) for m in ms]
    for c in range(K):
        y = scipy.signal.oaconvolve(x * np.exp(-2j * np.pi * ((c * n) % K) / K), taps.astype(np.float64))[:total]
        for o, m in zip(out, ms):
            o[c] = y[m]
    return out


def autocorr_model(x):
    """The reference's definition on the largest power of two: IFFT(|FFT(x)| / N), forward divided by N, inverse not."""
    N = 1 << (int(x.size).bit_length() - 1)
    return np.fft.ifft(np.abs(np.fft.fft(x[:N].astype(np.float64))) / N) * N


def first_max(v):
    best, top = 0, v[0]
    for i in range(1, v.size):
        if v[i] > top:
            best, top = i, v[i]
    return best


def scan_model(per_block, drops, fs, K):
    """The whole scan in float64 from the channelizer model's outputs: magnitudes, captures restarting at drops, running means
    over the detector's windows, first strict maximum, scores.  Returns (rounds, plots [K, flen + llen], records)."""
    lib = _native.lib()
    rate = 2 * fs // K
    size = lib.tsdrgpu_frd_capture_size(rate)
    w = [C.c_int() for _ in range(4)]
    lib.tsdrgpu_frd_windows(rate, *[C.byref(v) for v in w])
    fmin, fmax, lmin, lmax = (v.value for v in w)
    plots = np.zeros((K, (fmax - fmin) + (lmax - lmin)))
    buf = np.zeros((K, 0))
    rounds = 0
    for y, g in zip(per_block, drops):
        if g:
            buf = np.zeros((K, 0))
        buf = np.concatenate([buf, np.abs(y)], axis=1)
        while buf.shape[1] >= size:
            rounds += 1
            for c in range(K):
                r = np.abs(autocorr_model(buf[c, :size]))
                lags = np.concatenate([r[fmin:fmax], r[lmin:lmax]])
                plots[c] = (plots[c] * (rounds - 1) + lags) / rounds
            buf = buf[:, size:]
    recs = []
    for c in range(K):
        rec = {"offset_hz": offsets(fs, K)[c], "rate": rate, "captures": rounds}
        for name, v in (("frame", plots[c, : fmax - fmin]), ("line", plots[c, fmax - fmin:])):
            i = first_max(v)
            sd = v.std()
            rec[name + "_index"] = i
            rec[name + "_score"] = (v[i] - v.mean()) / sd if sd > 0 else 0.0
            srt = np.sort(v)
            rec[name + "_margin"] = (srt[-1] - srt[-2]) / max(abs(srt[-1]), 1e-300)
        fps, h = C.c_double(), C.c_int()
        lib.tsdrgpu_videomode_from_peaks(fmin, rec["frame_index"], lmin, rec["line_index"], rate, C.byref(fps), C.byref(h))
        rec["fps"], rec["height"] = fps.value, h.value
        recs.append(rec)
    return rounds, plots, recs, (fmin, fmax, lmin, lmax)


# the two-emitter use case: fs = 32 MS/s cut into K = 8 channels of 8 MS/s.  A = 62.5 Hz x 800 lines at +8 MHz (channel 2),
# B = 80 Hz x 1000 lines at -12 MHz (channel 5): both frame and line periods are whole samples at the channel rate (128000 / 160
# and 100000 / 100), so the detector's integer lags give the heights exactly.  A channel "holds" an emitter when its output band
# (centre +- fs / K) overlaps the emitter's occupied band (+- 0.4 bw around its offset); channels 0 and 7 hold neither.
UC_FS, UC_K, UC_SECS = 32_000_000, 8, 0.4
UC_A = dict(fv=62.5, h=800, offset=8_000_000.0, channel=2)
UC_B = dict(fv=80.0, h=1000, offset=-12_000_000.0, channel=5)
UC_BW = 3_000_000
# frame-plot scores of the float64 scan model on this capture (7 capture rounds): A 30.6, B 41.6, best of channels 0 / 7: 4.2; the
# model's peaks give 62.5 Hz x 800 and 80 Hz x 1000 exactly.  The test asks a factor 3 of the GPU scan
UC_FACTOR = 3.0


def uc_capture():
    n = int(UC_FS * UC_SECS)
    a, ra = emitter(n, UC_FS, UC_A["fv"], UC_A["h"], 11, 1.0, UC_A["offset"], UC_BW)
    b, rb = emitter(n, UC_FS, UC_B["fv"], UC_B["h"], 12, 1.5, UC_B["offset"], UC_BW)
    rng = np.random.default_rng(13)
    z = a + b + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return iq(z), ra, rb


def holds_neither(fs, K):
    out = []
    for c, off in enumerate(offsets(fs, K)):
        lo, hi = off - fs / K, off + fs / K
        hit = False
        for e in (UC_A, UC_B):
            for shift in (-fs, 0, fs):                     # the Nyquist channel wraps
                if lo < e["offset"] + 0.4 * UC_BW + shift and e["offset"] - 0.4 * UC_BW + shift < hi:
                    hit = True
        if not hit:
            out.append(c)
    return out


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("K,Q,fs", [(2, 4, 1_000_000), (8, 16, 8_000_000), (8, 32, 8_000_000), (64, 4, 64_000_000),
                                    (64, 16, 64_000_000), (256, 16, 64_000_000), (256, 32, 100_000_000)])
def test_stage_matches_float64_model(K, Q, fs):
    import torch
    from tempestsdr_b200 import api
    ctx = api.Context(0)
    ch = ctx.channelizer()
    ch.configure(fs, K, Q)
    taps = api.channelizer_design(fs, K, Q)
    offs = offsets(fs, K)
    tones = [(offs[1] + 0.1 * fs / K, 1.0), (offs[-1] - 0.3 * fs / K, 0.5), (offs[K // 2] + 0.2 * fs / K, 2.0), (0.37 * fs, 0.7)]
    z = tone_signal(300_000, fs, tones, seed=K + Q)
    rng = np.random.default_rng(K * 100 + Q)
    sizes = [0, 1, 17, int(rng.integers(1, 5000)), 3, 0, int(rng.integers(10_000, 90_000)), Q * K - 2, int(rng.integers(10_000, 90_000))]
    drops = [0, 0, 5, 0, 1234, 777, 0, K // 2 + 1, 3]               # block 5: empty, only a loss
    segs, got, o = [], [], 0
    for k, g in zip(sizes, drops):
        blk = z[o:o + k]; o += k
        segs.append((g, blk))
        out, od = ch.run(torch.from_numpy(iq(blk)).cuda(), g)
        got.append(out.cpu().numpy())
    want = channelizer_model(segs, taps, K)
    worst = []
    for c in range(K):
        peak = max((np.max(np.abs(w[c])) for w in want if w.shape[1]), default=0.0)
        err = max((float(np.max(np.abs(g_[c, :, 0] + 1j * g_[c, :, 1] - w[c]))) for g_, w in zip(got, want) if w.shape[1]), default=0.0)
        worst.append(err / peak)
    for g_, w in zip(got, want):
        assert g_.shape[:2] == w.shape
    print(f"K={K} Q={Q}: max error / channel peak = {max(worst):.2e}")
    assert max(worst) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("K", [4, 16, 64])
def test_every_channel_is_the_tuner_at_its_offset(K):
    import torch
    from tempestsdr_b200 import api
    fs, Q = 16_000_000, 16
    ctx = api.Context(0)
    ch = ctx.channelizer()
    ch.configure(fs, K, Q)
    z = tone_signal(200_000, fs, [(f, 1.0) for f in offsets(fs, K)[:: max(1, K // 8)] + 0.15 * fs / K], seed=K)
    blocks = [(0, 50_000), (300, 70_000), (0, 80_000)]
    x = torch.from_numpy(iq(z)).cuda()
    outs, o = [], 0
    for g, k in blocks:
        outs.append(ch.run(x[2 * o:2 * (o + k)], g)[0].cpu().numpy()); o += k
    got = np.concatenate(outs, axis=1)
    checked = 0
    for c, off in enumerate(offsets(fs, K)):
        if abs(off) + fs / (2 * K) > fs / 2:
            continue
        tn = ctx.tuner()
        tn.configure(fs, off, fs / K, K // 2, Q * K - 1)
        t_out, o = [], 0
        for g, k in blocks:
            t_out.append(cplx(tn.run(x[2 * o:2 * (o + k)], g)[0].cpu().numpy())); o += k
        want = np.concatenate(t_out)
        mine = got[c, :, 0] + 1j * got[c, :, 1]
        assert mine.size == want.size
        assert np.max(np.abs(mine - want)) <= 1e-5 * np.max(np.abs(want)), c
        checked += 1
    assert checked >= K - 1


@pytest.mark.gpu
@pytest.mark.parametrize("K,Q", [(8, 16), (64, 8), (256, 4)])
def test_magnitudes_and_block_cut_invariance(K, Q):
    """Magnitude mode is tsdrgpu_am_demod of the complex mode, bit for bit; the same stream cut three ways (drops at the same
    places) gives bit-identical outputs in both modes."""
    import torch
    from tempestsdr_b200 import api
    fs = 64_000_000
    ctx = api.Context(0)
    z = tone_signal(400_000, fs, [(f, 1.0) for f in offsets(fs, K)[::3] + 1e5], seed=Q)
    x_all = iq(z)
    drops_at = {50_000: 12, 120_003: 1, 300_000: 5000}
    rng = np.random.default_rng(K)
    results = []
    for cut in range(3):
        cm, cc = ctx.channelizer(), ctx.channelizer()
        cm.configure(fs, K, Q); cc.configure(fs, K, Q)
        small = [0, 1, K // 2 - 1, K // 2, Q * K - 2, Q * K - 1]
        bounds, o = [0], 0
        while o < z.size:
            k = int(rng.choice(small)) if rng.random() < 0.5 or cut == 0 else int(rng.integers(1, 60_000 if cut == 1 else 5_000))
            nxt = min(o + k, z.size)
            for d in sorted(drops_at):
                if o < d < nxt:
                    nxt = d
            bounds.append(nxt); o = nxt
        mags, cps, pending = [], [], dict(drops_at)
        for a, b in zip(bounds[:-1], bounds[1:]):
            g = pending.pop(a, 0)
            blk = torch.from_numpy(x_all[2 * a:2 * b].copy()).cuda()
            m, _ = cm.run(blk, g, magnitude=True)
            c, _ = cc.run(blk, g)
            mags.append(m.cpu().numpy()); cps.append(c.contiguous())
        mag = np.concatenate(mags, axis=1)
        cpl = torch.cat(cps, dim=1)
        demod = np.stack([ctx.am_demod(cpl[c].reshape(-1).contiguous()).cpu().numpy() for c in range(K)])
        assert np.array_equal(mag.view(np.uint32), demod.view(np.uint32))
        results.append((mag, cpl.cpu().numpy()))
    for m, c in results[1:]:
        assert m.shape == results[0][0].shape and np.array_equal(m.view(np.uint32), results[0][0].view(np.uint32))
        assert np.array_equal(c.view(np.uint32), results[0][1].view(np.uint32))


def _scan_signal(fs, secs, seed):
    """One raster at channel 2 of K = 8 (55-87 Hz, a height the detector can see) and a tone elsewhere, over noise."""
    n = int(fs * secs)
    a, _ = emitter(n, fs, 62.5, 800, seed, 1.0, 2 * fs / 8, fs / 8 * 0.75)
    rng = np.random.default_rng(seed)
    return a + 0.3 * np.exp(2j * np.pi * (-0.3) * np.arange(n)) + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))


@pytest.mark.gpu
def test_scan_matches_float64_model():
    import torch
    from tempestsdr_b200 import api
    fs, K, Q = 8_000_000, 8, 16
    ctx = api.Context(0)
    sc = ctx.scan()
    sc.configure(fs, K, Q)
    z = _scan_signal(fs, 1.0, 21)
    rng = np.random.default_rng(5)
    segs, drops, o = [], [], 0
    while o < z.size:
        k = min(int(rng.integers(1, 200_000)), z.size - o)
        g = int(rng.choice([0, 0, 0, 0, 0, 0, 0, 7, 3000]))
        segs.append((g, z[o:o + k])); drops.append(g); o += k
    segs.insert(10, (999, z[:0])); drops.insert(10, 999)               # an empty block that only reports a loss
    for g, b in segs:
        sc.run(torch.from_numpy(iq(b)).cuda(), g)
    recs = sc.records()
    plots, fl, ll = sc.plots()
    taps = api.channelizer_design(fs, K, Q)
    ys = channelizer_model([(g, cplx(iq(b))) for g, b in segs], taps, K)
    rounds, mplots, mrec, (fmin, fmax, lmin, lmax) = scan_model(ys, drops, fs, K)
    assert rounds >= 10 and all(r.captures == rounds for r in recs)
    assert (fl, ll) == (fmax - fmin, lmax - lmin)
    assert np.max(np.abs(plots - mplots)) <= 1e-4 * np.max(np.abs(mplots))
    d_plots = torch.from_numpy(plots).cuda()
    for c in range(K):
        r, m = recs[c], mrec[c]
        assert r.offset_hz == m["offset_hz"] and r.rate == m["rate"]
        for name in ("frame", "line"):
            assert abs(getattr(r, name + "_score") - m[name + "_score"]) <= 1e-4 * max(abs(m[name + "_score"]), 1.0), (c, name)
        if m["frame_margin"] > 1e-4 and m["line_margin"] > 1e-4:
            assert (r.frame_index, r.line_index) == (m["frame_index"], m["line_index"]), c
            assert (r.fps, r.height) == (m["fps"], m["height"]), c
        pk = (C.c_int32 * 2)()
        _native.check(ctx._lib.tsdrgpu_plot_peaks(ctx._h, ctx.stream, d_plots[c].data_ptr(), fl, d_plots[c].data_ptr() + 8 * fl, ll, pk))
        assert (pk[0], pk[1]) == (r.frame_index, r.line_index), c
    assert sc.results()[0]["channel"] == 2


@pytest.mark.gpu
def test_two_emitters_scan_then_tune():
    import torch
    from tempestsdr_b200 import api
    x, ra, rb = uc_capture()
    ctx = api.Context(0)
    sc = ctx.scan()
    sc.configure(UC_FS, UC_K)
    items = 1 << 20
    for k in range(0, x.size, items):
        sc.run(torch.from_numpy(x[k:k + items].copy()).cuda(), 0)
    table = sc.results()
    print("scan:", [(r["channel"], round(r["frame_score"], 2), round(r["fps"], 2), r["height"]) for r in table])
    top = {table[0]["channel"], table[1]["channel"]}
    assert top == {UC_A["channel"], UC_B["channel"]}
    by_ch = {r["channel"]: r for r in table}
    rate = 2 * UC_FS // UC_K
    worst_other = max(by_ch[c]["frame_score"] for c in holds_neither(UC_FS, UC_K))
    for e in (UC_A, UC_B):
        r = by_ch[e["channel"]]
        assert abs(rate / r["fps"] - rate / e["fv"]) <= 1.0 and r["height"] == e["h"], (e, r)
        assert r["frame_score"] >= UC_FACTOR * worst_other, (e, r, worst_other)
    # then tune to the top row and look at the picture
    top_row = table[0]
    own = ra if top_row["channel"] == UC_A["channel"] else rb
    p, g = _collect_pipeline(UC_FS, top_row["height"], top_row["fps"])
    p.set_tuner(top_row["offset_hz"], UC_FS / UC_K, UC_K // 2)
    items = 262144
    for k in range(0, x.size - items + 1, items):
        p.process(x[k:k + items].copy(), 0)
    p.flush()
    assert len(g["frames"]) >= 8
    c = [raster_corr(f, w, own) for w, f in g["frames"][-4:]]
    print("tuned to the top row:", c)
    assert min(v for v, _ in c) >= OWN_MIN and len({i for _, i in c}) == 1, c
    p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,tuned", [("float32", False), ("int8", False), ("float32", True), ("int8", True)])
def test_scan_does_not_disturb_the_pixel_path(fmt, tuned):
    import torch
    from tempestsdr_b200 import api, synth
    fs, h, fv, K, items, nblk = 8_000_000, 125, 60.0, 8, 65536, 40
    w = int(2 * fs / (fv * h))
    base = cplx(synth.video_like_iq(nblk * items // 2, fs, w, h, fv, seed=23))
    z = base + 0.3 * np.exp(2j * np.pi * 0.2 * np.arange(base.size))
    if fmt == "int8":
        data = np.clip(np.round(iq(z) * 40.0), -128, 127).astype(np.int8)
    else:
        data = iq(z)
    drops = {3: 3, 5: 40_001, 20: 1, 30: 2 * items}
    ctx = api.Context(0)
    sc = ctx.scan()
    sc.configure(fs, K, 0)
    runs = []
    for with_scan in (False, True):
        p, g = _collect_pipeline(fs, h, fv)
        if tuned:
            p.set_tuner(1_000_000, 2_000_000, 2)
        if with_scan:
            p.set_scan(K)
        for k in range(nblk):
            blk = data[k * items:(k + 1) * items].copy()
            d = drops.get(k, 0)
            if k == 25:
                p.process(np.zeros(0, np.float32), 999)
                if with_scan:
                    sc.run(torch.zeros(0, dtype=torch.float32, device="cuda"), 999)
            if fmt == "int8":
                p.process_raw(blk, d)
            else:
                p.process(blk, d)
            if with_scan:
                x = ctx.convert_samples(torch.from_numpy(blk).cuda()) if fmt == "int8" else torch.from_numpy(blk).cuda()
                sc.run(x, d)
        p.flush()
        runs.append((g, p.scan_results()))
        p.close()
    (g0, t0), (g1, t1) = runs
    assert t0 == [] and len(g0["frames"]) >= 3
    _same(g0, g1)
    assert t1[0]["captures"] >= 1
    assert t1 == sc.results()


@pytest.mark.gpu
def test_superbandwidth_mode_pauses_the_scan():
    from tempestsdr_b200 import synth
    fs, h, fv = 400_000, 80, 50.0
    items = 16384
    nblk = 2 * (4 * (10 * int(fs / fv) + int(0.5 * fs)) // (items // 2) + 8)
    x = synth.video_like_iq(nblk * items // 2, fs, 200, 80, fv, seed=41, snr_db=25)
    outs = []
    for scanning in (False, True):
        p, g = _collect_pipeline(fs, h, fv, on_retune=lambda off: None)
        if scanning:
            p.set_scan(2)
        p.set_param("superresolution", 1)
        for k in range(nblk):
            p.process(x[k * items:(k + 1) * items].copy(), 0)
        p.flush()
        outs.append((list(g["frames"]), p.scan_results()))
        if scanning:
            p.set_param("superresolution", 0)                  # the mode ends: the scan resumes from a clean start
            for k in range(60):
                p.process(x[k * items:(k + 1) * items].copy(), 0)
            p.flush()
            after = p.scan_results()
        p.close()
    (f0, _), (f1, t1) = outs
    assert len(f0) >= 4
    assert [w for w, _ in f0] == [w for w, _ in f1]
    for (_, a), (_, b) in zip(f0, f1):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert len(t1) == 2 and all(r["captures"] == 0 for r in t1)
    assert all(r["captures"] >= 1 for r in after)


@pytest.mark.gpu
def test_host_library_scan_file(tmp_path, monkeypatch):
    from tests.test_host_library import FRAME_CB, MINE, PLOT_CB, PLUGIN, VALUE_CB, bind
    x, _, _ = uc_capture()
    raw = tmp_path / "two.raw"
    x.tofile(raw)
    out = tmp_path / "scan.csv"
    got = []
    monkeypatch.setenv("TSDR_NO_DROP", "1")
    monkeypatch.setenv("TSDR_NO_RAW_SINK", "1")
    monkeypatch.setenv("TSDR_SCAN", "8")
    monkeypatch.setenv("TSDR_SCAN_FILE", str(out))
    lib = bind(MINE)
    t = C.c_void_p()
    nv, npl = VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
    fcb = FRAME_CB(lambda b, ww, hh, c: got.append(ww))
    lib.tsdr_init(C.byref(t), nv, npl, None)
    lib.tsdr_setresolution(t, UC_A["h"], UC_A["fv"]); lib.tsdr_motionblur(t, 0.0); lib.tsdr_setgain(t, 0.5)
    assert lib.tsdr_loadplugin(t, PLUGIN.encode(), f'"{raw}" {UC_FS} float'.encode()) == 0
    rc = []
    th = threading.Thread(target=lambda: rc.append(lib.tsdr_readasync(t, fcb, None)))
    th.start()
    deadline = time.time() + 120
    while len(got) < 30 and time.time() < deadline:            # 30 frames at 62.5 Hz: more than the 0.4 s recording
        time.sleep(0.05)
    assert lib.tsdr_stop(t) == 0
    th.join(timeout=60)
    assert rc == [0]
    lib.tsdr_free(C.byref(t))
    lines = out.read_text().strip().splitlines()
    assert lines[0] == "channel,offset_hz,rate,captures,fps,height,frame_score,line_score"
    rows = [dict(zip(lines[0].split(","), v.split(","))) for v in lines[1:]]
    assert len(rows) == 8
    scores = [float(r["frame_score"]) for r in rows]
    assert scores == sorted(scores, reverse=True)
    first = rows[0]
    e = UC_A if int(first["channel"]) == UC_A["channel"] else UC_B
    assert int(first["channel"]) == e["channel"] and int(first["captures"]) >= 5
    rate = 2 * UC_FS // UC_K
    assert int(first["height"]) == e["h"] and abs(rate / float(first["fps"]) - rate / e["fv"]) <= 1.0
