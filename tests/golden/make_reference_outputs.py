"""Records tests/golden/reference_outputs.json: what the REAL reference (oracle/_ref, compiled from the original sources by
`make -C oracle ref`) returns in every scenario that tests/test_oracle_pinning.py, tests/test_host_library.py and
tests/test_rawfile_plugin.py compare this project with.  Each scenario is the tests' own function, run here with the
reference's libraries in place of this project's; values are stored as tests/test_golden.py's `observed` makes them.

Run where the reference sources are present, after build():   python tests/golden/make_reference_outputs.py
"""
import itertools
import json
import os
import pathlib
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as orc                       # noqa: E402
from tests import test_host_library as H               # noqa: E402
from tests import test_oracle_pinning as P             # noqa: E402
from tests import test_rawfile_plugin as RF            # noqa: E402
from tests.test_golden import REFERENCE_OUTPUTS, observed   # noqa: E402


def parameter_sets(test):
    """Every parameter set pytest generates for `test` from its parametrize marks, as keyword dicts."""
    axes = []
    for mark in getattr(test, "pytestmark", []):
        if mark.name == "parametrize":
            names = [n.strip() for n in mark.args[0].split(",")]
            axes.append([dict(zip(names, v if len(names) > 1 else (v,))) for v in mark.args[1]])
    return [dict(kv for d in combo for kv in d.items()) for combo in itertools.product(*axes)]


def main():
    R = orc.ref()
    out = {}
    for name, fn in P.SCENARIOS.items():
        for params in parameter_sets(getattr(P, "test_" + name)):
            out[P.key(name, **params)] = [observed(v) for _, v in fn(R, **params)]

    tmp = pathlib.Path(tempfile.mkdtemp())
    out["host_library/exported"] = H.exported(orc.REF_LIB_SO, "tsdr_")
    out["host_library/status_codes"] = [observed(v) for _, v in H.status_codes(orc.REF_LIB_SO, orc.REF_RAWFILE_SO, tmp)]
    out["host_library/more_setter_scenarios"] = [observed(v) for _, v in H.more_setter_scenarios(orc.REF_LIB_SO, orc.REF_RAWFILE_SO, tmp)]

    plugin = RF.bind_plugin(orc.REF_RAWFILE_NOPACE_SO)
    out["rawfile_plugin/init_rc"] = [plugin.tsdrplugin_init(RF.C.create_string_buffer(p.encode())) for p in RF.PARAMS]
    for dtype, name in RF.DTYPES:
        raw = tmp / f"iq.{name}"
        RF.one_and_a_half_blocks(dtype, raw)
        out[f"rawfile_plugin/blocks/{name}"] = [observed(b) for b in RF.collect_blocks(orc.REF_RAWFILE_NOPACE_SO, f'"{raw}" 8000000 {name}', 4)]
    for dtype, name in RF.SINK_DTYPES:
        raw = tmp / f"q.{name}"
        fs, _, _ = RF.quantised_recording(dtype, raw)
        out[f"rawfile_plugin/recording/{name}"] = [observed(b) for b in RF.collect_blocks(orc.REF_RAWFILE_NOPACE_SO, f'"{raw}" {fs} {name}', 6)]

    with open(REFERENCE_OUTPUTS, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print(f"{REFERENCE_OUTPUTS}: {len(out)} scenarios, {os.path.getsize(REFERENCE_OUTPUTS)} bytes")


if __name__ == "__main__":
    np.seterr(all="ignore")
    main()
