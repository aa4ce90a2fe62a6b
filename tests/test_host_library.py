"""The C host library (tempestsdr_b200/lib/libTSDRLibrary.so): same exported tsdr_* symbols, status codes and
error-text behaviour as the reference library.  The reference's side of each comparison is what the compiled reference
library did in the same scenario with the reference's own RawFile source plugin, recorded in
tests/golden/reference_outputs.json; this library runs it with this project's RawFile plugin in its plain ten-symbol
mode (test_rawfile_plugin pins that plugin to the reference's).  CPU part here; the GPU end-to-end run is
test_host_library_end_to_end (marked gpu)."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile
import threading
import time

import numpy as np
import pytest

from oracle import oracle as orc
from tempestsdr_b200 import synth
from tests.test_golden import assert_matches_reference, reference_outputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MINE = os.path.join(ROOT, "tempestsdr_b200", "lib", "libTSDRLibrary.so")
PLUGIN = os.path.join(ROOT, "tempestsdr_b200", "lib", "TSDRPlugin_RawFileGPU.so")

FRAME_CB = C.CFUNCTYPE(None, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_void_p)
VALUE_CB = C.CFUNCTYPE(None, C.c_int, C.c_double, C.c_double, C.c_void_p)
PLOT_CB = C.CFUNCTYPE(None, C.c_int, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_uint32, C.c_void_p)


def bind(path):
    lib = C.CDLL(path)
    lib.tsdr_init.argtypes = [C.POINTER(C.c_void_p), VALUE_CB, PLOT_CB, C.c_void_p]
    lib.tsdr_setresolution.argtypes = [C.c_void_p, C.c_int, C.c_double]
    lib.tsdr_motionblur.argtypes = [C.c_void_p, C.c_float]
    lib.tsdr_setgain.argtypes = [C.c_void_p, C.c_float]
    lib.tsdr_setparameter_int.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    lib.tsdr_setparameter_double.argtypes = [C.c_void_p, C.c_int, C.c_double]
    lib.tsdr_loadplugin.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
    lib.tsdr_readasync.argtypes = [C.c_void_p, FRAME_CB, C.c_void_p]
    lib.tsdr_sync.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.tsdr_getlasterrortext.argtypes = [C.c_void_p]
    lib.tsdr_getlasterrortext.restype = C.c_char_p
    for f in ("tsdr_stop", "tsdr_isrunning", "tsdr_unloadplugin", "tsdr_getsamplerate"):
        getattr(lib, f).argtypes = [C.c_void_p]
    lib.tsdr_free.argtypes = [C.POINTER(C.c_void_p)]
    lib.tsdr_setbasefreq.argtypes = [C.c_void_p, C.c_uint32]
    return lib


def exported(path, prefix):
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    return sorted(l.split()[-1] for l in out.splitlines() if l.split()[-1].startswith(prefix))


def plugin_error_text(plugin, params, tmp_path):
    """The text `plugin` itself reports when its init rejects `params`: run on a private copy of it, so that the copy the
    library loads keeps its own state (a plugin keeps its state in statics)."""
    copy = os.path.join(tempfile.mkdtemp(dir=tmp_path), os.path.basename(plugin))     # a fresh file: a loaded one is never overwritten
    shutil.copy(plugin, copy)
    lib = C.CDLL(copy)
    lib.tsdrplugin_getlasterrortext.restype = C.c_char_p
    assert lib.tsdrplugin_init(C.create_string_buffer(params.encode())) != 0      # a plugin may tokenise its parameters in place
    return lib.tsdrplugin_getlasterrortext()


def forwarded(text, plugin_text):
    """A library hands a plugin's rejection text on to the host: that text is the plugin's own, so what is compared is that
    it was forwarded unchanged."""
    return "<the plugin's own error text>" if text == plugin_text else text


def test_same_exported_api_as_the_reference_library():
    assert exported(MINE, "tsdr_") == reference_outputs("host_library/exported")
    assert len(exported(MINE, "tsdr_")) == 18


def status_codes(path, plugin, tmp_path):
    """Status codes and error texts of one library through a fixed sequence of calls, `plugin` as the source plugin."""
    raw = tmp_path / "iq.raw"
    synth.noise_iq(4096, seed=1).tofile(raw)
    nv, npl = VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
    lib = bind(path)
    t = C.c_void_p()
    lib.tsdr_init(C.byref(t), nv, npl, None)
    lib.tsdr_setresolution(t, 525, 60.0); lib.tsdr_motionblur(t, 0.0); lib.tsdr_setgain(t, 0.5)
    r = []
    r.append(("readasync without plugin", (lib.tsdr_readasync(t, FRAME_CB(lambda *a: None), None), lib.tsdr_getlasterrortext(t))))
    r.append(("unload without plugin", (lib.tsdr_unloadplugin(t), lib.tsdr_getlasterrortext(t))))
    r.append(("getsamplerate without plugin", (lib.tsdr_getsamplerate(t), lib.tsdr_getlasterrortext(t))))
    r.append(("bad resolution", (lib.tsdr_setresolution(t, 0, 60.0), lib.tsdr_getlasterrortext(t))))
    r.append(("bad param id", (lib.tsdr_setparameter_int(t, 99, 1), lib.tsdr_getlasterrortext(t))))
    r.append(("good param", (lib.tsdr_setparameter_int(t, 0, 1), lib.tsdr_getlasterrortext(t))))
    r.append(("bad double id", (lib.tsdr_setparameter_double(t, 7, 1.0), lib.tsdr_getlasterrortext(t))))
    r.append(("bad motionblur", (lib.tsdr_motionblur(t, 1.5), None)))
    r.append(("missing plugin file", (lib.tsdr_loadplugin(t, b"/nonexistent/plugin.so", b""), lib.tsdr_getlasterrortext(t))))
    r.append(("not a plugin", (lib.tsdr_loadplugin(t, orc.PORT_SO.encode(), b""), lib.tsdr_getlasterrortext(t))))
    bad = f'"{raw}" 8000000'
    r.append(("plugin param error", (lib.tsdr_loadplugin(t, plugin.encode(), bad.encode()), forwarded(lib.tsdr_getlasterrortext(t), plugin_error_text(plugin, bad, tmp_path)))))
    r.append(("plugin ok", (lib.tsdr_loadplugin(t, plugin.encode(), f'"{raw}" 8000000 float'.encode()), lib.tsdr_getlasterrortext(t))))
    r.append(("getsamplerate", (lib.tsdr_getsamplerate(t), lib.tsdr_getlasterrortext(t))))
    r.append(("sync too far", (lib.tsdr_sync(t, 100000, 1), lib.tsdr_getlasterrortext(t))))
    r.append(("sync ok", (lib.tsdr_sync(t, 3, 3), lib.tsdr_getlasterrortext(t))))
    r.append(("isrunning", (lib.tsdr_isrunning(t), None)))
    r.append(("stop when idle", (lib.tsdr_stop(t), lib.tsdr_getlasterrortext(t))))
    r.append(("unload", (lib.tsdr_unloadplugin(t), lib.tsdr_getlasterrortext(t))))
    lib.tsdr_free(C.byref(t))
    assert not t.value
    return r


def test_status_codes_and_error_text_match_the_reference(tmp_path):
    assert_matches_reference("host_library/status_codes", status_codes(MINE, PLUGIN, tmp_path))


def more_setter_scenarios(path, plugin, tmp_path):
    """Second sweep of the boundary (TSDRLibrary.c:136-262, 420-560): every setter with in-range, edge and out-of-range values, before
    and after a plugin is loaded, repeated loads / unloads."""
    raw = tmp_path / "iq.raw"
    synth.noise_iq(4096, seed=2).tofile(raw)
    nv, npl = VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
    lib = bind(path)
    t = C.c_void_p()
    lib.tsdr_init(C.byref(t), nv, npl, None)
    r = []
    txt = lambda: lib.tsdr_getlasterrortext(t)
    r.append(("fresh: error text", (None, txt())))
    r.append(("isrunning fresh", (lib.tsdr_isrunning(t), None)))
    r.append(("setbasefreq without plugin", (lib.tsdr_setbasefreq(t, 100_000_000), txt())))
    r.append(("setgain without plugin", (lib.tsdr_setgain(t, 0.5), txt())))
    r.append(("sync before resolution", (lib.tsdr_sync(t, 1, 0), txt())))
    for h, fv in ((525, 60.0), (1125, 59.94), (-3, 60.0), (525, 0.0), (525, -1.0), (1, 1.0)):
        r.append((f"setresolution {h} {fv}", (lib.tsdr_setresolution(t, h, fv), txt())))
    lib.tsdr_setresolution(t, 525, 60.0)
    for mb in (0.0, 0.5, 1.0, -0.1, 1.0001):
        r.append((f"motionblur {mb}", (lib.tsdr_motionblur(t, mb), txt())))
    for pid in range(-1, 11):
        r.append((f"param_int {pid}", (lib.tsdr_setparameter_int(t, pid, 1), txt())))
        lib.tsdr_setparameter_int(t, pid, 0)
    for pid in range(-1, 4):
        r.append((f"param_double {pid}", (lib.tsdr_setparameter_double(t, pid, 0.25), txt())))
    r.append(("plugin ok", (lib.tsdr_loadplugin(t, plugin.encode(), f'"{raw}" 8000000 float'.encode()), txt())))
    r.append(("error text after success", (None, txt())))
    r.append(("plugin again", (lib.tsdr_loadplugin(t, plugin.encode(), f'"{raw}" 2000000 int8'.encode()), txt())))
    r.append(("getsamplerate", (lib.tsdr_getsamplerate(t), txt())))
    for g in (0.0, 1.0, -0.5, 1.5):
        r.append((f"setgain {g}", (lib.tsdr_setgain(t, g), txt())))
    r.append(("setbasefreq", (lib.tsdr_setbasefreq(t, 433_920_000), txt())))
    for px, d in ((0, 0), (5, 0), (5, 1), (5, 2), (5, 3), (5, 4), (-5, 0), (10_000_000, 2), (10_000_000, 0)):
        r.append((f"sync {px} {d}", (lib.tsdr_sync(t, px, d), txt())))
    r.append(("bad plugin params keep", (lib.tsdr_loadplugin(t, plugin.encode(), b"nofile 0 float"),
                                         forwarded(txt(), plugin_error_text(plugin, "nofile 0 float", tmp_path)))))
    r.append(("getsamplerate after failed load", (lib.tsdr_getsamplerate(t), txt())))
    r.append(("unload", (lib.tsdr_unloadplugin(t), txt())))
    r.append(("unload twice", (lib.tsdr_unloadplugin(t), txt())))
    r.append(("stop idle", (lib.tsdr_stop(t), txt())))
    lib.tsdr_free(C.byref(t))
    return r


def test_more_setter_scenarios_match_the_reference(tmp_path):
    """Status codes and error texts identical to the compiled reference's in more_setter_scenarios."""
    assert_matches_reference("host_library/more_setter_scenarios", more_setter_scenarios(MINE, PLUGIN, tmp_path))


def test_readasync_without_gpu_fails_loudly(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    raw = tmp_path / "iq.raw"
    synth.noise_iq(1 << 20, seed=1).tofile(raw)
    lib = bind(MINE)
    t = C.c_void_p()
    nv, npl = VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
    lib.tsdr_init(C.byref(t), nv, npl, None)
    lib.tsdr_setresolution(t, 525, 60.0)
    assert lib.tsdr_loadplugin(t, PLUGIN.encode(), f'"{raw}" 8000000 float nopace'.encode()) == 0
    rc = lib.tsdr_readasync(t, FRAME_CB(lambda *a: None), None)
    assert rc == 6                                        # TSDR_CANNOT_OPEN_DEVICE
    assert b"no CPU fallback" in lib.tsdr_getlasterrortext(t)
    assert lib.tsdr_isrunning(t) == 0
    lib.tsdr_free(C.byref(t))


@pytest.mark.gpu
def test_host_library_end_to_end(tmp_path, monkeypatch):
    """tsdr_readasync + a RawFile plugin on a file (this project's, in plain ten-symbol mode: float samples handed over
    on the host like the reference's plugin does): delivered frames equal the oracle's stage-wise replay."""
    from tests.test_pipeline_gpu import run_oracle_stream
    O = orc.best()
    fs, h, fv = 2_000_000, 125, 60.0
    w, _, _ = O.geometry(fs, h, fv)
    items = 512 * 1024                                    # SAMPLES_TO_READ_AT_ONCE of the plugin
    nblk = 6
    iq = synth.video_like_iq(nblk * items // 2, fs, w, h, fv, seed=31)
    raw = tmp_path / "iq.raw"
    iq.tofile(raw)
    _, want = run_oracle_stream(O, [iq[k * items:(k + 1) * items] for k in range(nblk)], fs, h, fv)
    got = []
    os.environ["TSDR_NO_DROP"] = "1"
    monkeypatch.setenv("TSDR_NO_RAW_SINK", "1")
    lib = bind(MINE)
    t = C.c_void_p()
    nv, npl = VALUE_CB(lambda *a: None), PLOT_CB(lambda *a: None)
    fcb = FRAME_CB(lambda b, ww, hh, c: got.append(np.ctypeslib.as_array(b, shape=(ww * hh,)).copy()))
    lib.tsdr_init(C.byref(t), nv, npl, None)
    lib.tsdr_setresolution(t, h, fv); lib.tsdr_motionblur(t, 0.0); lib.tsdr_setgain(t, 0.5)
    for pid, v in ((0, 1), (1, 0), (6, 1)):
        lib.tsdr_setparameter_int(t, pid, v)
    assert lib.tsdr_loadplugin(t, PLUGIN.encode(), f'"{raw}" {int(fs)} float'.encode()) == 0
    rc = []
    th = threading.Thread(target=lambda: rc.append(lib.tsdr_readasync(t, fcb, None)))
    th.start()
    deadline = time.time() + 60
    while len(got) < len(want) and time.time() < deadline:     # the plugin loops over the file; first pass is enough
        time.sleep(0.05)
    assert lib.tsdr_isrunning(t) == 1
    assert lib.tsdr_stop(t) == 0
    th.join(timeout=30)
    assert rc == [0] and lib.tsdr_isrunning(t) == 0
    assert len(got) >= len(want) > 3
    for k, wv in enumerate(want):
        assert np.array_equal(got[k].view(np.uint32), wv.view(np.uint32)), f"frame {k}"
    lib.tsdr_free(C.byref(t))


@pytest.mark.gpu
def test_a_plain_c_host_delivers_frames_on_the_gpu(tmp_path):
    """The same C host, as a GPU test: on the B200 it has to deliver frames (rc = 0), not merely fail politely."""
    import torch
    assert torch.cuda.is_available()
    test_a_plain_c_host_links_and_runs(tmp_path)


def test_a_plain_c_host_links_and_runs(tmp_path):
    """INTEGRATION.md section A, literally: a C program compiled against include/TSDRLibrary.h and linked with libTSDRLibrary.a +
    libtsdrgpu.so drives init -> setresolution -> loadplugin -> readasync -> free.  On this machine's hardware it must either
    deliver frames (GPU) or fail with TSDR_CANNOT_OPEN_DEVICE and the 'no CPU fallback' text (no GPU)."""
    import subprocess
    libdir = os.path.join(ROOT, "tempestsdr_b200", "lib")
    exe = tmp_path / "host_smoke"
    subprocess.run(["gcc", "-O1", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c_host", "host_smoke.c"),
                    os.path.join(libdir, "libTSDRLibrary.a"), "-L", libdir, "-ltsdrgpu", f"-Wl,-rpath,{libdir}", "-ldl", "-lpthread", "-lm",
                    "-o", str(exe)], check=True)
    raw = tmp_path / "iq.int8"
    (np.random.default_rng(3).integers(-100, 100, 4 << 20, dtype=np.int64).astype(np.int8)).tofile(raw)
    plugin = os.path.join(libdir, "TSDRPlugin_RawFileGPU.so")
    r = subprocess.run([str(exe), plugin, f'"{raw}" 2000000 int8 nopace'], capture_output=True, text=True, timeout=120,
                       env=dict(os.environ, TSDR_NO_DROP="1"))
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr[-500:])
    import torch
    if torch.cuda.is_available():
        assert "rc=0" in r.stdout
    else:
        assert "rc=6" in r.stdout and "no CPU fallback" in r.stdout
    # and a plugin that does not exist is reported like the reference does (TSDR_INCOMPATIBLE_PLUGIN = 7)
    r = subprocess.run([str(exe), "/nonexistent/plugin.so", "x"], capture_output=True, text=True, timeout=60)
    assert "loadplugin rc=7" in r.stdout
