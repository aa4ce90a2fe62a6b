"""The GPU-aware RawFile front end (tempestsdr_b200/plugins) and the raw-sample ingest behind it (SURVEY section 8f-1).

CPU: the plugin is an ordinary ten-symbol TSDR plugin -- same parameter errors as the reference's TSDRPlugin_RawFile, the
same floats through the ordinary callback (including what is delivered around the end of the file).
GPU: the device conversion is bit-identical to the plugin's host expressions for EVERY 8- and 16-bit code, and a run
through the host library with the raw sink delivers bit-identical frames to a run that converts on the host, fed the
floats the reference's own plugin delivers for the same recording.
What the reference's plugin did is recorded in tests/golden/reference_outputs.json (tests/golden/make_reference_outputs.py)."""
import ctypes as C
import os
import subprocess
import threading
import time

import numpy as np
import pytest

from oracle import oracle as orc
from tempestsdr_b200 import synth
from tests.test_golden import assert_matches_reference, reference_outputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLUGIN = os.path.join(ROOT, "tempestsdr_b200", "lib", "TSDRPlugin_RawFileGPU.so")
MINE = os.path.join(ROOT, "tempestsdr_b200", "lib", "libTSDRLibrary.so")
PLUGIN_CB = C.CFUNCTYPE(None, C.POINTER(C.c_float), C.c_uint64, C.c_void_p, C.c_int64)
TEN = ["tsdrplugin_init", "tsdrplugin_getsamplerate", "tsdrplugin_getName", "tsdrplugin_setsamplerate", "tsdrplugin_setbasefreq",
       "tsdrplugin_stop", "tsdrplugin_setgain", "tsdrplugin_readasync", "tsdrplugin_getlasterrortext", "tsdrplugin_cleanup"]


def reference_floats(raw: np.ndarray) -> np.ndarray:
    """TSDRPlugin_RawFile.c:241-261 restated: double quotient, then rounded to float."""
    v = raw.astype(np.float64)
    if raw.dtype == np.int8: return (v / 128.0).astype(np.float32)
    if raw.dtype == np.uint8: return ((v - 128) / 128.0).astype(np.float32)
    if raw.dtype == np.int16: return (v / 32767.0).astype(np.float32)
    if raw.dtype == np.uint16: return ((v - 32767) / 32767.0).astype(np.float32)
    return raw.astype(np.float32)


def bind_plugin(path):
    lib = C.CDLL(path)
    lib.tsdrplugin_init.argtypes = [C.c_char_p]; lib.tsdrplugin_init.restype = C.c_int
    lib.tsdrplugin_getlasterrortext.restype = C.c_char_p
    lib.tsdrplugin_getsamplerate.restype = C.c_uint32
    lib.tsdrplugin_readasync.argtypes = [PLUGIN_CB, C.c_void_p]; lib.tsdrplugin_readasync.restype = C.c_int
    lib.tsdrplugin_getName.argtypes = [C.c_char_p]
    return lib


def collect_blocks(path, params, nblocks):
    """Drive a plugin like a host would, without any library: the first `nblocks` blocks it delivers."""
    lib = bind_plugin(path)
    assert lib.tsdrplugin_init(C.create_string_buffer(params.encode())) == 0, lib.tsdrplugin_getlasterrortext()
    got = []

    def cb(buf, items, ctx, dropped):
        if len(got) < nblocks:
            got.append(np.ctypeslib.as_array(buf, shape=(items,)).copy())
        if len(got) >= nblocks:
            lib.tsdrplugin_stop()
    fn = PLUGIN_CB(cb)
    assert lib.tsdrplugin_readasync(fn, None) == 0
    lib.tsdrplugin_cleanup()
    return got


def test_plugin_exports_the_plugin_abi():
    out = subprocess.run(["nm", "-D", "--defined-only", PLUGIN], capture_output=True, text=True, check=True).stdout
    syms = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert set(TEN) <= syms
    assert syms - set(TEN) == {"tsdrpluginx_set_raw_sink"}          # the one documented, optional extra (include/TSDRPluginX.h)
    lib = bind_plugin(PLUGIN)
    name = C.create_string_buffer(256)
    lib.tsdrplugin_getName(name)
    assert b"Raw" in name.value


PARAMS = ["", "somefile", "somefile 0 float", "somefile 8000000", "somefile 8000000 int12", "somefile -5 int8",
          "somefile 2000000000 float", "'some file' 8000000 float"]


@pytest.mark.parametrize("params", PARAMS)
def test_parameter_errors_match_the_reference_plugin(params):
    mine = bind_plugin(PLUGIN)
    rc = mine.tsdrplugin_init(C.create_string_buffer(params.encode()))
    ok_expected = params.endswith("8000000 float")
    assert (rc == 0) == ok_expected
    assert rc in (0, 4)                                    # TSDR_PLUGIN_PARAMETERS_WRONG
    assert (mine.tsdrplugin_getlasterrortext() is None) == (rc == 0)
    assert reference_outputs("rawfile_plugin/init_rc")[PARAMS.index(params)] == rc
    assert mine.tsdrplugin_init(C.create_string_buffer(b"f 1000 int8 nopace block=7")) == 4      # odd block
    assert mine.tsdrplugin_init(C.create_string_buffer(b"f 1000 int8 bogus")) == 4
    assert mine.tsdrplugin_init(C.create_string_buffer(b"f 1000 int8 nopace block=4096")) == 0
    assert mine.tsdrplugin_getsamplerate() == 1000


def one_and_a_half_blocks(dtype, path):
    """A recording of one and a half plugin blocks of seeded samples; returns the samples."""
    items = 512 * 1024
    rng = np.random.default_rng(5)
    n = items + items // 2
    if dtype == np.float32:
        data = rng.standard_normal(n).astype(np.float32)
    else:
        info = np.iinfo(dtype)
        data = rng.integers(info.min, info.max + 1, n, dtype=np.int64).astype(dtype)
    data.tofile(path)
    return data


DTYPES = [(np.int8, "int8"), (np.uint8, "uint8"), (np.int16, "int16"), (np.uint16, "uint16"), (np.float32, "float")]


@pytest.mark.parametrize("dtype,name", DTYPES)
def test_plugin_without_a_sink_is_an_ordinary_rawfile_plugin(tmp_path, dtype, name):
    """No raw sink offered (as under the reference library): host conversion, float callback, and the reference's behaviour
    at the end of the file -- the block buffer is delivered as it stands (fresh head, stale tail), then the file restarts."""
    items = 512 * 1024
    raw = tmp_path / f"iq.{name}"
    data = one_and_a_half_blocks(dtype, raw)
    mine = collect_blocks(PLUGIN, f'"{raw}" 8000000 {name} nopace', 4)
    conv = reference_floats(data)
    second = np.concatenate([conv[items:], conv[items // 2: items]])       # 0.5 block fresh + the stale tail of block 1
    want = [conv[:items], second, conv[:items], second]
    for k in range(4):
        assert np.array_equal(mine[k].view(np.uint32), want[k].view(np.uint32)), f"block {k}"
    assert_matches_reference(f"rawfile_plugin/blocks/{name}", [(f"block {k}", mine[k]) for k in range(4)])


# ------------------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.int8, np.uint8, np.int16, np.uint16])
def test_device_conversion_is_exact_for_every_code(dtype):
    import torch
    from tempestsdr_b200.api import Context
    gpu = Context(0)
    info = np.iinfo(dtype)
    codes = np.arange(info.min, info.max + 1, dtype=np.int64).astype(dtype)
    codes = np.concatenate([codes, codes[::-1], codes[:3]])                 # odd length: exercises the scalar tail
    tdt = {np.int8: torch.int8, np.uint8: torch.uint8, np.int16: torch.int16, np.uint16: torch.uint16}[dtype]
    d = torch.from_numpy(codes.view(np.int8 if dtype == np.uint8 else (np.int16 if dtype == np.uint16 else dtype))).cuda().view(tdt)
    got = gpu.convert_samples(d).cpu().numpy()
    want = reference_floats(codes)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def _run_host_library(plugin_path, params, fs, h, fv, nframes, env=None):
    from tests.test_host_library import bind, FRAME_CB, VALUE_CB, PLOT_CB
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    os.environ["TSDR_NO_DROP"] = "1"
    try:
        got = []
        lib = bind(MINE)
        t = C.c_void_p()
        nv, npl = VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
        fcb = FRAME_CB(lambda b, ww, hh, c: got.append(np.ctypeslib.as_array(b, shape=(ww * hh,)).copy()))
        lib.tsdr_init(C.byref(t), nv, npl, None)
        lib.tsdr_setresolution(t, h, fv); lib.tsdr_motionblur(t, 0.0); lib.tsdr_setgain(t, 0.5)
        for pid, v in ((0, 1), (1, 0), (6, 1)):
            lib.tsdr_setparameter_int(t, pid, v)
        assert lib.tsdr_loadplugin(t, plugin_path.encode(), params.encode()) == 0, lib.tsdr_getlasterrortext(t)
        rc = []
        th = threading.Thread(target=lambda: rc.append(lib.tsdr_readasync(t, fcb, None)))
        th.start()
        deadline = time.time() + 60
        while len(got) < nframes and time.time() < deadline:
            time.sleep(0.02)
        assert lib.tsdr_stop(t) == 0
        th.join(timeout=30)
        assert rc == [0]
        lib.tsdr_free(C.byref(t))
        return got
    finally:
        for k, v in old.items():
            if v is None: os.environ.pop(k, None)
            else: os.environ[k] = v


def quantised_recording(dtype, path):
    """Six plugin blocks of video-like IQ at 2 MS/s, quantised to `dtype`; returns (fs, h, fv)."""
    fs, h, fv = 2_000_000, 125, 60.0
    w, _, _ = orc.port().geometry(fs, h, fv)
    items = 512 * 1024
    iq = synth.video_like_iq(6 * items // 2, fs, w, h, fv, seed=77)
    info = np.iinfo(dtype)
    scale = 100.0 if dtype != np.int16 else 20000.0
    q = np.clip(np.round(iq / np.abs(iq).max() * scale) + (128 if dtype == np.uint8 else 0), info.min, info.max).astype(dtype)
    q.tofile(path)
    return fs, h, fv


SINK_DTYPES = [(np.int8, "int8"), (np.uint8, "uint8"), (np.int16, "int16")]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,name", SINK_DTYPES)
def test_raw_sink_run_equals_a_run_with_the_reference_plugin(tmp_path, dtype, name):
    """Same recording, same library: (a) the GPU-aware plugin with the sink withheld, converting on the host -- the floats it
    hands over for the whole recording are the reference RawFile plugin's, bit for bit -- and (b) the GPU-aware plugin with
    its raw sink (samples cross PCIe as integers).  Frames agree bit for bit -- the device conversion is the host
    conversion."""
    raw = tmp_path / f"iq.{name}"
    fs, h, fv = quantised_recording(dtype, raw)
    blocks = collect_blocks(PLUGIN, f'"{raw}" {fs} {name} nopace', 6)
    assert_matches_reference(f"rawfile_plugin/recording/{name}", [(f"block {k}", b) for k, b in enumerate(blocks)])
    nframes = 12
    a = _run_host_library(PLUGIN, f'"{raw}" {fs} {name} nopace', fs, h, fv, nframes, env={"TSDR_NO_RAW_SINK": "1"})
    b = _run_host_library(PLUGIN, f'"{raw}" {fs} {name} nopace', fs, h, fv, nframes)
    assert min(len(a), len(b)) >= nframes
    for k in range(nframes):
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), f"frame {k}: raw sink vs host conversion"
