"""The tuner (digital down-converter ahead of the pixel path, csrc/tuner.cu): filter design and count arithmetic on the host,
the kernel against a float64 model, block-cut invariance, the pipeline as the composition "tuner, then the untuned pipeline at
fs/D", the two-emitter use case, live reconfiguration, and the host library's TSDR_TUNER knob."""
import ctypes as C
import os
import threading
import time

import numpy as np
import pytest
import scipy.signal

from tempestsdr_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BETA = 0.1102 * (80.0 - 8.7)


def design(fs, off, bw, D=1, ntaps=0):
    lib = _native.lib()
    taps = np.zeros(1023, np.float32)
    n, inc = C.c_int(0), C.c_uint64(0)
    rc = lib.tsdrgpu_tuner_design(fs, off, bw, D, ntaps, taps.ctypes.data_as(C.c_void_p), 1023, C.byref(n), C.byref(inc))
    return rc, taps[: n.value], inc.value


# ---------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("fs,bw,ntaps", [(8_000_000, 2_000_000, 65), (100_000_000, 25_000_000, 0), (25_000_000, 1_000_000, 1023),
                                         (2_000_000, 1_999_999, 3), (48_000, 6_000, 129), (200_000_000, 3_125_000, 0),
                                         (10_000_000, 2_500_000, 17), (64_000_000, 1_000_000, 257)])
def test_design_matches_firwin(fs, bw, ntaps):
    rc, taps, inc = design(fs, 0.0, bw, 1, ntaps)
    assert rc == 0
    n = ntaps or min(16 * int(np.ceil(fs / bw)) + 1, 1023)
    want = scipy.signal.firwin(n, bw / 2, window=("kaiser", BETA), fs=fs)
    assert taps.size == n and np.max(np.abs(taps.astype(np.float64) - want)) <= 1e-7
    assert inc == 0


def test_default_ntaps_rule_and_phase_increment():
    # 16 * ceil(fs / bandwidth) + 1, at most 1023
    for fs, bw, want in [(100_000_000, 25_000_000, 65), (8_000_000, 3_000_000, 49), (8_000_000, 8_000_000, 17),
                         (8_000_000, 1_000_000, 129), (100_000_000, 1_000_000, 1023), (62_000_000, 1_000_000, 993)]:
        assert design(fs, 0.0, bw, 1, 0)[1].size == want, (fs, bw)
    for fs, off in [(8_000_000, 1_000_000.0), (8_000_000, -2_500_000.0), (100_000_000, 12_345_678.0), (3, 1.0)]:
        _, _, inc = design(fs, off, 1.0, 1, 0)
        want = int(round(off / fs * 2.0 ** 64)) % 2 ** 64
        assert abs(((inc - want + 2 ** 63) % 2 ** 64) - 2 ** 63) <= 2 ** 11, (fs, off)       # round() in 64-bit long double


@pytest.mark.parametrize("cfg,text", [
    ((8_000_000, 0.0, 1e6, 0, 0), "decimation must be an integer in 1..64"),
    ((8_000_000, 0.0, 1e6, 65, 0), "decimation must be an integer in 1..64"),
    ((8_000_000, 0.0, 1e6, 1, 2), "ntaps must be odd, in 3..1023"),
    ((8_000_000, 0.0, 1e6, 1, 1025), "ntaps must be odd, in 3..1023"),
    ((8_000_000, 0.0, 1e6, 1, 1), "ntaps must be odd, in 3..1023"),
    ((8_000_000, 0.0, 0.0, 1, 0), "bandwidth_hz must be > 0"),
    ((8_000_000, 0.0, -5.0, 1, 0), "bandwidth_hz must be > 0"),
    ((8_000_000, 0.0, 1e6, 3, 0), "multiple of the decimation (fs % D == 0)"),
    ((8_000_000, 0.0, 2_000_001, 4, 0), "must not exceed the decimated rate (bandwidth <= fs / D)"),
    ((8_000_000, 3_500_001, 1e6, 1, 0), "inside the capture (|offset| + bandwidth / 2 <= fs / 2)"),
    ((8_000_000, -3_600_000, 1e6, 4, 0), "inside the capture (|offset| + bandwidth / 2 <= fs / 2)"),
])
def test_invalid_configurations_are_rejected_with_their_rule(cfg, text):
    lib = _native.lib()
    assert lib.tsdrgpu_tuner_design(*cfg, None, 0, None, None) == -3          # TSDRGPU_EINVAL
    assert text in lib.tsdrgpu_last_error(None).decode()
    assert lib.tsdrgpu_tuner_design(8_000_000, 3_500_000.0, 1e6, 4, 0, None, 0, None, None) == 0     # the edges are allowed


def test_out_pairs_matches_a_model():
    lib = _native.lib()
    rng = np.random.default_rng(7)

    def ceil_div(a, b):
        return -(-a // b)

    o, od = C.c_uint64(0), C.c_uint64(0)
    for seq in range(1000):
        D = int(rng.choice([1, 2, 3, 4, 7, 8, 64]))
        pos = 0
        for _ in range(20):
            k = int(rng.choice([0, 1, D - 1, D, D + 1, int(rng.integers(0, 100_000))]))
            g = int(rng.choice([0, 0, 0, 1, D - 1, int(rng.integers(0, 5000)), 2 ** 40 + int(rng.integers(0, 999))]))
            assert lib.tsdrgpu_tuner_out_pairs(pos, k, g, D, C.byref(o), C.byref(od)) == 0
            assert od.value == ceil_div(pos + g, D) - ceil_div(pos, D), (seq, pos, k, g, D)
            assert o.value == ceil_div(pos + g + k, D) - ceil_div(pos + g, D), (seq, pos, k, g, D)
            pos += g + k
    assert lib.tsdrgpu_tuner_out_pairs(0, 1, 0, 0, C.byref(o), C.byref(od)) == -3


def test_host_library_rejects_a_malformed_tuner_knob(tmp_path, monkeypatch):
    """TSDR_TUNER is checked before any device work: a malformed or invalid value fails tsdr_readasync with
    TSDR_INVALID_PARAMETER_VALUE and a text naming what is wrong."""
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
    for value, text in [("abc", b"TSDR_TUNER: expected"), ("1e6", b"TSDR_TUNER: expected"), ("1e6,2e6,4,65,9", b"TSDR_TUNER: expected"),
                        ("1e6,2e6,", b"TSDR_TUNER: expected"), ("1e6,2e6,2.5", b"TSDR_TUNER: expected"),
                        ("0,3e6,4", b"bandwidth <= fs / D"), ("3.5e6,2e6,4", b"|offset| + bandwidth / 2 <= fs / 2"), ("0,1e6,3", b"fs % D == 0")]:
        monkeypatch.setenv("TSDR_TUNER", value)
        assert lib.tsdr_readasync(t, FRAME_CB(lambda *a: None), None) == 9, value        # TSDR_INVALID_PARAMETER_VALUE
        assert text in lib.tsdr_getlasterrortext(t), value
        assert lib.tsdr_isrunning(t) == 0
    lib.tsdr_free(C.byref(t))


# ---------------------------------------------------------------------------------------------------------------- GPU helpers

def model(segments, taps, inc, D):
    """float64 model: zero-fill every gap, mix with the integer phase, filter, decimate, keep the outputs inside blocks.
    segments: [(dropped_before, complex block)].  Returns the outputs block by block."""
    total = sum(g + b.size for g, b in segments)
    x = np.zeros(total, np.complex128)
    spans, pos = [], 0
    for g, b in segments:
        pos += g
        x[pos:pos + b.size] = b
        spans.append((pos, b.size))
        pos += b.size
    n = np.arange(total, dtype=np.uint64)
    ph = (n * np.uint64(inc)).view(np.int64).astype(np.float64)
    x *= np.exp(-1j * np.pi * ph / 2.0 ** 63)
    y = scipy.signal.oaconvolve(x, taps.astype(np.float64))[:total]
    out = []
    for b0, k in spans:
        m0, m1 = -(-b0 // D), -(-(b0 + k) // D)
        out.append(y[np.arange(m0, m1, dtype=np.int64) * D])
    return out


def iq(z):
    out = np.empty(2 * z.size, np.float32)
    out[0::2], out[1::2] = z.real, z.imag
    return out


def cplx(f):
    return f[0::2].astype(np.float64) + 1j * f[1::2].astype(np.float64)


def tone_signal(n, fs, tones, seed, noise=0.3):
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    z = noise * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    for f, a in tones:
        z = z + a * np.exp(2j * np.pi * f / fs * t + 1j * rng.uniform(0, 6.28))
    return z


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("fs,off,bw,D,ntaps,fmt", [
    (8_000_000, 1_500_000.0, 2_000_000, 4, 0, "float32"),
    (8_000_000, -2_750_000.0, 1_000_000, 8, 0, "float32"),
    (9_000_000, -1_000_000.0, 3_000_000, 3, 1023, "float32"),
    (8_000_000, 0.0, 8_000_000, 1, 17, "float32"),
    (10_000_000, 2_345_678.5, 4_000_000, 2, 257, "int8"),
    (8_000_000, -1_234_567.0, 500_000, 8, 1023, "int8"),
    (64_000_000, 7_000_000.0, 1_000_000, 64, 0, "float32"),
])
def test_stage_matches_float64_model(fs, off, bw, D, ntaps, fmt):
    import torch
    from tempestsdr_b200 import api
    ctx = api.Context(0)
    tn = ctx.tuner()
    tn.configure(fs, off, bw, D, ntaps)
    taps, inc = tn.taps, tn.phase_inc
    rng = np.random.default_rng(D * 1000 + len(taps))
    z = tone_signal(400_000, fs, [(off + 0.2 * bw, 1.0), (off - 0.3 * bw, 0.5), (-off, 2.0)], seed=D)
    sizes = [0, 1, 17, 70_000, 3, 0, 100_000, 129_000, 101_000]
    drops = [0, 0, 5, 0, 1234, 777, 0, D + 1, 3]
    segs, got, gotd, o = [], [], [], 0
    for k, g in zip(sizes, drops):
        blk = z[o:o + k]; o += k
        if fmt == "int8":
            q = np.clip(np.round(iq(blk) * 30.0), -128, 127).astype(np.int8)
            x = ctx.convert_samples(torch.from_numpy(q).cuda())
            blk = cplx((q.astype(np.float64) / 128.0).astype(np.float32))
        else:
            x = torch.from_numpy(iq(blk)).cuda()
        segs.append((g, blk))
        out, od = tn.run(x, g)
        got.append(out.cpu().numpy()); gotd.append(od)
    want = model(segs, taps, inc, D)
    peak = max(np.max(np.abs(w)) for w in want if w.size)
    worst = 0.0
    for k, (g_, w) in enumerate(zip(got, want)):
        assert g_.size == 2 * w.size, k
        if w.size:
            worst = max(worst, float(np.max(np.abs(cplx(g_) - w))))
    pos = 0
    for (g, b), od in zip(segs, gotd):
        assert od == -(-(pos + g) // D) - (-(-pos // D)); pos += g + b.size
    print(f"D={D} ntaps={len(taps)} {fmt}: max error / peak = {worst / peak:.2e}")
    assert worst <= 1e-5 * peak


@pytest.mark.gpu
@pytest.mark.parametrize("D,ntaps", [(1, 33), (3, 65), (8, 1023)])
def test_block_cut_invariance(D, ntaps):
    """The same stream (drops at the same places) cut three ways -- sizes 0, 1, D-1, ntaps-2 and random -- gives bit-identical
    outputs and the same output drop counts."""
    import torch
    from tempestsdr_b200 import api
    fs = 24_000_000
    ctx = api.Context(0)
    z = tone_signal(300_000, fs, [(2e6, 1.0)], seed=ntaps)
    x_all = iq(z)
    drops_at = {50_000: 12, 120_003: 1, 200_000: 5000}          # absolute input index (data only) -> lost pairs before it
    rng = np.random.default_rng(D)
    results = []
    for cut in range(3):
        tn = ctx.tuner()
        tn.configure(fs, -3e6, fs // D if D > 1 else 4e6, D, ntaps)
        small = [0, 1, max(D - 1, 0), ntaps - 2]
        bounds, o = [0], 0
        while o < z.size:
            k = int(rng.choice(small)) if rng.random() < 0.5 or cut == 0 else int(rng.integers(1, 40_000 if cut == 1 else 3_000))
            nxt = min(o + k, z.size)
            for d in sorted(drops_at):                       # a drop always starts a block
                if o < d < nxt:
                    nxt = d
            bounds.append(nxt); o = nxt
        outs, ods, pending = [], [], dict(drops_at)
        for a, b in zip(bounds[:-1], bounds[1:]):
            g = pending.pop(a, 0)                            # a drop goes with the first block (possibly empty) at its index
            out, od = tn.run(torch.from_numpy(x_all[2 * a:2 * b].copy()).cuda(), g)
            outs.append(out.cpu().numpy()); ods.append(od)
        assert not pending
        results.append((np.concatenate(outs), sum(ods)))
    for r in results[1:]:
        assert r[0].size == results[0][0].size and np.array_equal(r[0].view(np.uint32), results[0][0].view(np.uint32))
        assert r[1] == results[0][1]


def _collect_pipeline(fs, h, fv, **kw):
    from tempestsdr_b200 import pipeline
    got = {"frames": [], "plots": [], "values": []}
    p = pipeline.Pipeline(samplerate=fs, height=h, refreshrate=fv, batch_frames=1, block_when_busy=True,
                          params={"autoshift": 1, "lowpass_before_sync": 1},
                          on_frame=lambda f, ww, hh: got["frames"].append((ww, f.copy())),
                          on_plot=lambda pid, off, v, sr: got["plots"].append((pid, off, sr, v.copy())),
                          on_value=lambda vid, a, b: got["values"].append((vid, a, b)), **kw)
    return p, got


def _same(a, b):
    assert len(a["frames"]) == len(b["frames"]) and len(a["plots"]) == len(b["plots"])
    for k, ((wa, fa), (wb, fb)) in enumerate(zip(a["frames"], b["frames"])):
        assert wa == wb and np.array_equal(fa.view(np.uint32), fb.view(np.uint32)), f"frame {k}"
    for k, (x, y) in enumerate(zip(a["plots"], b["plots"])):
        assert x[:3] == y[:3] and np.array_equal(x[3].view(np.uint64), y[3].view(np.uint64)), f"plot {k}"
    assert a["values"] == b["values"]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["small_int8", "cfg2_100MSps"])
def test_pipeline_is_the_tuner_then_the_untuned_pipeline(shape):
    """A tuned pipeline delivers exactly what an untuned pipeline at fs/D delivers when it is fed, block by block, the
    stage-level tuner's output and output drop counts: frames, plots and values bit-identical, with drops in the stream."""
    import torch
    from tempestsdr_b200 import api, synth
    if shape == "small_int8":
        fs, D, h, fv, off, bw, items, nblk = 8_000_000, 4, 125, 60.0, 1_500_000.0, 2_000_000, 65536, 44
    else:
        fs, D, h, fv, off, bw, items, nblk = 100_000_000, 4, 1125, 60.0, -20_000_000.0, 25_000_000, 512 * 1024, 44
    fsi = fs // D
    wi = int(2 * fsi / (fv * h))
    base = synth.video_like_iq(nblk * items // 2, fsi, wi, h, fv, seed=17, carrier_hz=0.0)
    up = np.repeat(cplx(base), D)[: nblk * items // 2]             # the raster at fs, shifted to the tuned band
    z = up * np.exp(2j * np.pi * off / fs * np.arange(up.size)) + 0.2 * np.exp(-2j * np.pi * 0.3 * np.arange(up.size))
    if shape == "small_int8":
        data = np.clip(np.round(iq(z) * 60.0), -128, 127).astype(np.int8)
        as_float = lambda b: (b.astype(np.float64) / 128.0).astype(np.float32)
    else:
        data = iq(z)
        as_float = lambda b: b
    drops = {3: 3, 5: 40_001, 6: 1, 40: 123_457, 42: 2 * items}    # blocks 7..39: two captures (small), five frames (cfg2)
    p1, g1 = _collect_pipeline(fs, h, fv)
    p1.set_tuner(off, bw, D)
    p2, g2 = _collect_pipeline(fsi, h, fv)
    ctx = api.Context(0)
    tn = ctx.tuner()
    tn.configure(fs, off, bw, D)
    for k in range(nblk):
        blk = data[k * items:(k + 1) * items].copy()
        d = drops.get(k, 0)
        if k == 41:                                                  # an empty block that only reports a loss
            p1.process(np.zeros(0, np.float32), 999)
            out, od = tn.run(torch.zeros(0, dtype=torch.float32, device="cuda"), 999)
            p2.process(out.cpu().numpy(), od)
        if shape == "small_int8":
            p1.process_raw(blk, d)
        else:
            p1.process(blk, d)
        out, od = tn.run(torch.from_numpy(as_float(blk)).cuda(), d)
        p2.process(out.cpu().numpy(), od)
    p1.flush(); p2.flush()
    assert p1.geometry()[0] == wi == p2.geometry()[0]
    assert len(g1["frames"]) >= 3 and (shape != "small_int8" or len(g1["plots"]) >= 2)
    _same(g1, g2)
    p1.close(); p2.close()


def emitter(n, fs, fv, h, seed, level, offset, bw):
    """One band-limited raster emitter at `offset`: the raster as 2 pixels per sample of fs_display = bw (the geometry rule),
    low-passed to bw in the test, shifted to offset.  Returns (complex samples at fs, raster h x w)."""
    rng = np.random.default_rng(seed)
    w = int(2 * bw / (fv * h))
    frame = np.full((h, w), 0.05)
    aw, ah = int(w * 0.85), int(h * 0.94)
    tiles = rng.uniform(0.35, 1.0, size=((ah + 7) // 8, (aw + 7) // 8))
    frame[:ah, :aw] = np.kron(tiles, np.ones((8, 8)))[:ah, :aw]
    t = np.arange(n)
    amp = frame.reshape(-1)[np.floor(t * (w * h * fv / fs)).astype(np.int64) % frame.size]
    spec = np.fft.fft(amp)
    f = np.fft.fftfreq(n, 1.0 / fs)
    spec[np.abs(f) > 0.4 * bw] = 0.0
    return level * np.fft.ifft(spec) * np.exp(2j * np.pi * offset / fs * t), frame


def raster_corr(frame, fw, raster):
    """Peak of the normalised circular cross-correlation of a delivered frame (fw pixels wide) with a raster's picture (its
    tiles, zero-mean, blanking zeroed: every raster has the same blanking layout, only the picture tells two emitters apart),
    resampled to the frame's size, and where it peaks.  A noiseless copy of the raster itself scores 0.56, another raster 0.06."""
    h, w = raster.shape
    fh = frame.size // fw
    r = raster[(np.arange(fh) * h // fh)][:, (np.arange(fw) * w // fw)]
    act = r != 0.05
    a = frame.reshape(fh, fw) - frame.mean(); b = np.where(act, r - r[act].mean(), 0.0)
    c = np.real(np.fft.ifft2(np.fft.fft2(a) * np.conj(np.fft.fft2(b)))) / (np.linalg.norm(a) * np.linalg.norm(b) + 1e-30)
    i = int(np.argmax(c))
    return float(c.reshape(-1)[i]), i


def two_emitters(fs=8_000_000, secs=0.5, seed=5):
    n = int(fs * secs)
    a, ra = emitter(n, fs, 60.0, 125, seed, 1.0, 2_000_000.0, 2_000_000)
    b, rb = emitter(n, fs, 50.0, 100, seed + 1, 3.0, -2_000_000.0, 2_000_000)
    rng = np.random.default_rng(seed + 2)
    z = a + b + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return iq(z), ra, rb


# thresholds of the use case (raster_corr's scale: 0.56 for a perfect copy, 0.06 for the other raster): a tuned pipeline's last
# frames correlate with their own emitter's picture at >= 0.3 and with the other one at <= 0.15, at one alignment in all of
# them (the sync detector has locked); the untuned pipeline stays below 0.2 on the weaker emitter
OWN_MIN, OTHER_MAX, UNTUNED_MAX = 0.3, 0.15, 0.2


@pytest.mark.gpu
def test_two_emitters_one_capture_two_pipelines():
    fs = 8_000_000
    x, ra, rb = two_emitters(fs)
    items = 65536
    pa, ga = _collect_pipeline(fs, 125, 60.0)
    pb, gb = _collect_pipeline(fs, 100, 50.0)
    pu, gu = _collect_pipeline(fs, 125, 60.0)
    pa.set_tuner(2_000_000, 2_000_000, 4)
    pb.set_tuner(-2_000_000, 2_000_000, 4)
    for k in range(x.size // items):
        blk = x[k * items:(k + 1) * items].copy()
        for p in (pa, pb, pu):
            p.process(blk, 0)
    for p in (pa, pb, pu):
        p.flush()
    res = {}
    for name, g, own, other in (("A", ga, ra, rb), ("B", gb, rb, ra)):
        assert len(g["frames"]) >= 8, name
        last = g["frames"][-4:]
        res[name] = ([raster_corr(f, w, own) for w, f in last], [raster_corr(f, w, other)[0] for w, f in last])
    cu = [raster_corr(f, w, ra)[0] for w, f in gu["frames"][-4:]]
    print(f"two emitters: tuned A {res['A']}, tuned B {res['B']}, untuned vs A {cu}")
    for name, (own, other) in res.items():
        assert min(c for c, _ in own) >= OWN_MIN and len({i for _, i in own}) == 1, (name, own)
        assert max(other) <= OTHER_MAX, (name, other)
    assert max(cu) < UNTUNED_MAX
    for p in (pa, pb, pu):
        p.close()


@pytest.mark.gpu
def test_live_reconfiguration_and_switching_off():
    """Retuning mid-run changes the geometry at the next block without an error; switching the tuner off gives frames
    bit-identical to a never-tuned pipeline fed the rest of the stream."""
    from tempestsdr_b200 import synth
    fs, h, fv = 8_000_000, 125, 60.0
    items = 65536
    x = synth.video_like_iq(60 * items // 2, fs, int(2 * fs / (fv * h)), h, fv, seed=9)
    p, g = _collect_pipeline(fs, h, fv)
    p.set_tuner(1_000_000, 2_000_000, 4)
    w_full = int(2 * fs / (fv * h))
    for k in range(20):
        p.process(x[k * items:(k + 1) * items].copy(), 0)
        if k == 0:
            assert p.geometry()[0] == w_full // 4
    p.set_tuner(-500_000, 1_000_000, 8)
    assert p.geometry()[0] == w_full // 4                 # takes effect at the next process() call
    p.process(x[20 * items:21 * items].copy(), 0)
    assert p.geometry()[0] == w_full // 8
    p.set_tuner(0, 0)                                     # off
    for k in range(21, 60):
        p.process(x[k * items:(k + 1) * items].copy(), 0)
    p.flush()
    assert p.geometry()[0] == w_full
    q, gq = _collect_pipeline(fs, h, fv)
    for k in range(21, 60):
        q.process(x[k * items:(k + 1) * items].copy(), 0)
    q.flush()
    after = [(w, f) for w, f in g["frames"] if w == w_full]
    assert len(after) == len(gq["frames"]) >= 3
    for (wa, fa), (wb, fb) in zip(after, gq["frames"]):
        assert np.array_equal(fa.view(np.uint32), fb.view(np.uint32))
    with pytest.raises(_native.TsdrGpuError, match="fs % D == 0"):
        p.set_tuner(0, 1_000_000, 3)
    with pytest.raises(_native.TsdrGpuError, match="bandwidth <= fs / D"):
        p.set_tuner(0, 2_000_000, 4)
        p.set_samplerate(4_000_000)
    p.close(); q.close()


@pytest.mark.gpu
def test_superbandwidth_mode_bypasses_the_tuner():
    from tempestsdr_b200 import synth
    fs, h, fv = 400_000, 80, 50.0
    items = 16384
    nblk = 2 * (4 * (10 * int(fs / fv) + int(0.5 * fs)) // (items // 2) + 8)
    x = synth.video_like_iq(nblk * items // 2, fs, 200, 80, fv, seed=41, snr_db=25)
    outs = []
    for tuned in (False, True):
        p, g = _collect_pipeline(fs, h, fv, on_retune=lambda off: None)
        if tuned:
            p.set_tuner(50_000, 100_000, 4)
        p.set_param("superresolution", 1)
        for k in range(nblk):
            p.process(x[k * items:(k + 1) * items].copy(), 0)
        p.flush()
        outs.append(g)
        p.close()
    assert len(outs[0]["frames"]) >= 4
    assert [w for w, _ in outs[0]["frames"]] == [w for w, _ in outs[1]["frames"]]
    for (_, a), (_, b) in zip(outs[0]["frames"], outs[1]["frames"]):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.gpu
def test_host_library_tuner_knob_shows_the_tuned_emitter(tmp_path, monkeypatch):
    from tests.test_host_library import FRAME_CB, MINE, PLOT_CB, PLUGIN, VALUE_CB, bind
    fs, D = 8_000_000, 4
    x, ra, rb = two_emitters(fs, secs=0.4)
    raw = tmp_path / "two.raw"
    x.tofile(raw)
    got = []
    monkeypatch.setenv("TSDR_NO_DROP", "1")
    monkeypatch.setenv("TSDR_NO_RAW_SINK", "1")
    monkeypatch.setenv("TSDR_TUNER", "2000000,2000000,4")
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
    c = [raster_corr(f, w, ra)[0] for w, f in got[8:12]]
    assert min(c) >= OWN_MIN, c
    lib.tsdr_free(C.byref(t))
