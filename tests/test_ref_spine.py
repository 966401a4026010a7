# SPDX-License-Identifier: Apache-2.0
"""The reference's OWN C++ spine observers (BaseOrientation -> FloorContact / WheelContact -> WheelOdometry) and
wheel_balancer controllers (WheelStopper -> WheelBalancer), compiled unmodified into oracle/_ref/ against stand-in
Eigen / palimpsest / spdlog headers (oracle/Makefile `ref`, oracle/ref_spine_shim.cpp), versus the oracle's
restatement and the kernels' arithmetic.

* tests/golden/ref_spine_runs.json holds that library's outputs on the seeded inputs of
  tests/golden/ref_spine_inputs.py: the comparison runs everywhere, reference tree or not;
* where oracle/_ref/libupkie_ref_spine.so exists (the build container, and the GPU box through the snapshot) the
  library itself is driven side by side with the oracle on fresh random inputs.
Rows a14 and f2 of SURVEY.md section 8."""
import ctypes as C
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import ref_spine_inputs as inputs  # noqa: E402
from test_controllers import OracleBalancer  # noqa: E402
from test_observers import OracleObservers  # noqa: E402
from upkie_b200 import _abi as A  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_spine_runs.json")


@pytest.fixture(scope="module")
def golden():
    return json.load(open(GOLDEN))


def _controller_columns(res):
    return [res[2, 1], res[2, 2], res[5, 1], res[5, 2], res[0, 3], res[0, 4], res[4, 3]]


@pytest.mark.parametrize("stream", [0, 1])
def test_observer_pipeline_matches_the_reference_cpp(golden, model, oracle_lib, stream):
    g = golden["observers"][stream]
    cfg = A.default_observer_config(model, float(g["spine_frequency"]))
    oo = OracleObservers(oracle_lib, cfg, 1)
    rows = inputs.observer_inputs(A, stream)
    ref = np.asarray(g["out"])
    keep = g["columns"]
    flags = [keep.index(A.OBSV_CONTACT), keep.index(A.OBSV_WHEEL_CONTACT), keep.index(A.OBSV_WHEEL_CONTACT + 1)]
    for k in range(inputs.N_STEPS):
        out = oo.step(rows[k:k + 1])[0]
        assert np.array_equal(out[keep][flags], ref[k][flags]), k  # contact decisions: exact
        assert np.allclose(out[keep], ref[k], rtol=1e-12, atol=1e-12), (k, np.abs(out[keep] - ref[k]).max())
        if k < 12:
            assert np.allclose(out[A.OBSV_ROT:A.OBSV_ROT + 9], g["rotation_first_steps"][k], rtol=0, atol=1e-14)
    assert 0.2 < ref[:, flags[0]].mean() < 0.95  # the sequence has both touchdowns and lift-offs
    oo.reset()
    assert np.allclose(oo.step(rows[0:1])[0][keep], g["first_after_reset"], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("stream", [0, 1])
def test_wheel_balancer_pipeline_matches_the_reference_cpp(golden, oracle_lib, stream):
    g = golden["controllers"][stream]
    cfg = A.default_wheel_balancer_config(float(g["spine_frequency"]))
    ob = OracleBalancer(oracle_lib, cfg, 1)
    ref = np.asarray(g["out"])
    for k, (obs3, target, act) in enumerate(inputs.controller_inputs(stream)):
        res, _ = ob.step(obs3.reshape(1, 3), None if target is None else target.reshape(1, 2), act.reshape(1, 6, 6))
        res = res.reshape(6, 6)
        assert np.isnan(res[2, 0]) and np.isnan(res[5, 0])
        assert np.allclose(_controller_columns(res), ref[k], rtol=1e-12, atol=1e-12), (k, _controller_columns(res), ref[k])
    assert {4.0, 2.0} <= set(ref[:, 4])  # both the turning and the straight gain scale occur
    assert (np.abs(ref[:, 0] - ref[:, 2]) > 1.0).any()  # the balancer really commands the wheels


@pytest.mark.parametrize("stream", [0, 1])
def test_kernel_arithmetic_matches_the_reference_cpp(golden, model, stream):
    """fp32 code of the kernels (CPU build) on the same inputs: observers and controllers."""
    from hostsim_wrap import lib, wheel_balancer_step

    g = golden["observers"][stream]
    cfg = A.default_observer_config(model, float(g["spine_frequency"]))
    L = lib()
    fp = C.POINTER(C.c_float)
    L.hostsim_observers_create.restype = C.c_void_p
    L.hostsim_observers_create.argtypes = [C.POINTER(A.UpkieObserverConfig), C.c_int]
    L.hostsim_observers_step.argtypes = [C.c_void_p, fp, fp]
    h = L.hostsim_observers_create(C.byref(cfg), 1)
    rows = inputs.observer_inputs(A, stream).astype(np.float32)
    ref = np.asarray(g["out"])
    keep = g["columns"]
    flags = [keep.index(A.OBSV_CONTACT), keep.index(A.OBSV_WHEEL_CONTACT), keep.index(A.OBSV_WHEEL_CONTACT + 1)]
    mismatches = 0
    for k in range(inputs.N_STEPS):
        out = np.zeros((1, A.OBSV_DIM), dtype=np.float32)
        L.hostsim_observers_step(h, rows[k:k + 1].ctypes.data_as(fp), out.ctypes.data_as(fp))
        mine = out[0][keep].astype(np.float64)
        mismatches += int(not np.array_equal(mine[flags], ref[k][flags]))
        cont = [i for i in range(len(keep)) if i not in flags]
        assert np.allclose(mine[cont], ref[k][cont], rtol=2e-4, atol=2e-4), (k, np.abs(mine[cont] - ref[k][cont]).max())
    assert mismatches <= 2  # a threshold crossing may land one cycle apart in fp32

    gc = golden["controllers"][stream]
    wcfg = A.default_wheel_balancer_config(float(gc["spine_frequency"]))
    state = np.zeros((1, 4), dtype=np.float32)
    refc = np.asarray(gc["out"])
    for k, (obs3, target, act) in enumerate(inputs.controller_inputs(stream)):
        a32 = act.astype(np.float32).reshape(1, 6, 6)
        wheel_balancer_step(wcfg, state, obs3.reshape(1, 3), None if target is None else target.reshape(1, 2), a32)
        assert np.allclose(_controller_columns(a32[0].astype(np.float64)), refc[k], rtol=1e-4, atol=2e-3), k


def test_reference_library_side_by_side(model, oracle_lib):
    """Whole observer rows and whole controller outputs versus the compiled reference (inputs other than the golden
    ones above): its outputs stored in tests/golden/ref_spine_side_by_side.json (every `every`-th step), and the
    library itself, step by step, where oracle/_ref/ exists."""
    O = oracle_lib
    side = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_spine_side_by_side.json")))
    freq, stream, every = side["spine_frequency"], side["stream"], side["every"]
    ocfg = A.default_observer_config(model, float(freq))
    wcfg = A.default_wheel_balancer_config(float(freq))
    ref = O.RefSpine(ocfg, wcfg, freq) if os.path.exists(O.REF_SPINE_PATH) else None
    oo = OracleObservers(oracle_lib, ocfg, 1)
    ob = OracleBalancer(oracle_lib, wcfg, 1)
    rows = inputs.observer_inputs(A, stream)
    for k in range(inputs.N_STEPS):
        mine = oo.step(rows[k:k + 1])[0]
        if k % every == 0:
            assert np.allclose(mine, side["observers"][k // every], rtol=1e-12, atol=1e-12), k
        if ref is not None:
            assert np.allclose(mine, ref.observers_step(rows[k]), rtol=1e-12, atol=1e-12), k
    for k, (obs3, target, act) in enumerate(inputs.controller_inputs(stream)):
        mine, _ = ob.step(obs3.reshape(1, 3), None if target is None else target.reshape(1, 2), act.reshape(1, 6, 6))
        if k % every == 0:
            stored = np.array([np.nan if v is None else v for v in side["controllers"][k // every]]).reshape(6, 6)
            assert np.allclose(mine.reshape(6, 6), stored, rtol=1e-12, atol=1e-12, equal_nan=True), k
        if ref is not None:
            theirs = ref.controllers_step(obs3, target, act)
            assert np.allclose(mine.reshape(6, 6), theirs, rtol=1e-12, atol=1e-12, equal_nan=True), k
