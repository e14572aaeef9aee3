"""The shipped Cython fast path (SURVEY.md section 8 row N1): host/py_corona_sim_b200.pyx = the reference's own binding
(included from its tree, every method unchanged) + Pyobservation_fit_b200, whose hot methods take buffers as typed
memoryviews and run without the GIL.  Built by oracle/build_pyx.py; the GPU box uses the prebuilt module."""
import glob
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("B200RT_REFERENCE")     # the reference's source tree, where one is at hand
OUT = os.path.join(ROOT, "oracle", "_ref", "py_corona_sim_fast")


def built():
    if REF and os.path.exists(os.path.join(REF, "python", "py_corona_sim.pyx")):
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import build_pyx
        build_pyx.build(verbose=False, fast=True)
    return bool(glob.glob(os.path.join(OUT, "py_corona_sim_gpu*.so")))


def test_fast_binding_builds_and_keeps_the_reference_class():
    if not built():
        pytest.skip("oracle/_ref/py_corona_sim_fast not built (needs B200RT_REFERENCE; python oracle/build_pyx.py)")
    code = ("import sys; sys.path.insert(0, %r); import py_corona_sim_gpu as m; "
            "assert issubclass(m.Pyobservation_fit_b200, m.Pyobservation_fit); "
            "print(len([x for x in dir(m.Pyobservation_fit) if not x.startswith('_')]))" % OUT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert int(r.stdout.strip()) >= 45          # every public method of the reference class is still there


@pytest.mark.gpu
def test_fast_binding_on_the_device():
    if not built():
        pytest.skip("oracle/_ref/py_corona_sim_fast not built")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "pyx_fast_worker.py"), "200000"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    out = json.loads(line[len("RESULT "):])
    assert out["brightness_shape"] == [2, 20000] and out["iph_shape"] == [2, 20000]
    assert out["brightness_max_rel"] < 1e-12 and out["col_dens_max_rel"] < 1e-12 and out["iph_equal"] and out["finite"]
    # ingest: the reference binding's Python loops cost seconds per 1e6 lines of sight; the buffer path tens of ms
    assert out["add_observation_s_per_1e6_fast_binding"] < 0.25
    assert out["add_observation_s_per_1e6_fast_binding"] * 10 < out["add_observation_s_per_1e6_reference_binding"]
    assert out["ticks_during_call"] > out["ticks_expected_if_released"]      # the GIL was released during the calls
