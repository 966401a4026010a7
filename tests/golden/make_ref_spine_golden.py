#!/usr/bin/env python
# SPDX-License-Identifier: Apache-2.0
"""Golden sequences of the reference's OWN C++ spine observers and wheel_balancer controllers.

Run in the build container:  python tests/golden/make_ref_spine_golden.py

``oracle/_ref/libupkie_ref_spine.so`` is the reference's upkie/cpp/observers/*.cpp and upkie/cpp/controllers/*.cpp
compiled unmodified and in place (oracle/Makefile ``ref``; Eigen / palimpsest / spdlog replaced by the stand-in
headers of oracle/standin/), behind the flat-array glue of oracle/ref_spine_shim.cpp. This script drives it with
seeded inputs and stores inputs + outputs in tests/golden/ref_spine_runs.json (and whole output rows of the
side-by-side run in tests/golden/ref_spine_side_by_side.json), so that the oracle's restatement
(ObserverPipelineOracle, WheelBalancerOracle) stays pinned on machines where the reference tree, and therefore the
library, are absent.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_spine_runs.json")
OUT_SIDE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_spine_side_by_side.json")
SIDE_BY_SIDE_EVERY = 4
sys.path.insert(0, ROOT)


def main():
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import ref_spine_inputs as inputs
    from oracle import oracle as O
    from upkie_b200 import _abi as A
    from upkie_b200.model import Model

    assert O.build_ref(), "oracle/_ref/libupkie_ref_spine.so could not be built (reference tree absent?)"
    model = Model.standard_upkie()
    out = {"generator": "tests/golden/make_ref_spine_golden.py", "inputs": "tests/golden/ref_spine_inputs.py",
           "observers": [], "controllers": []}
    keep = [A.OBSV_PITCH, A.OBSV_ANGVEL, A.OBSV_ANGVEL + 1, A.OBSV_ANGVEL + 2, A.OBSV_CONTACT, A.OBSV_WHEEL_CONTACT,
            A.OBSV_WHEEL_CONTACT + 1, A.OBSV_LEG_TORQUE, A.OBSV_WHEEL_INERTIA, A.OBSV_WHEEL_INERTIA + 1, A.OBSV_ODOM_POS,
            A.OBSV_ODOM_VEL]
    for stream, freq in enumerate((1000, 250)):
        oc = A.default_observer_config(model, float(freq))
        ref = O.RefSpine(oc, None, freq)
        rows = inputs.observer_inputs(A, stream)
        outs = np.array([ref.observers_step(r) for r in rows])
        ref.reset()
        after_reset = ref.observers_step(rows[0])
        out["observers"].append({"spine_frequency": freq, "columns": keep, "out": outs[:, keep].tolist(),
                                 "rotation_first_steps": outs[:12, A.OBSV_ROT:A.OBSV_ROT + 9].tolist(),
                                 "first_after_reset": after_reset[keep].tolist()})
        print("observers", freq, "contact fraction", outs[:, A.OBSV_CONTACT].mean(), "final odometry", outs[-1, A.OBSV_ODOM_POS])
    for stream, freq in enumerate((1000, 200)):
        oc = A.default_observer_config(model, 1000.0)
        wc = A.default_wheel_balancer_config(float(freq))
        ref = O.RefSpine(oc, wc, freq)
        rows = []
        for obs3, target, act in inputs.controller_inputs(stream):
            res = ref.controllers_step(obs3, target, act)
            unchanged = np.array_equal(res[[0, 1, 3, 4]][:, [0, 1, 2, 5]], act[[0, 1, 3, 4]][:, [0, 1, 2, 5]]) and \
                np.array_equal(res[[2, 5]][:, 3:], act[[2, 5]][:, 3:])
            assert unchanged  # the pipeline only touches wheel position / velocity / feedforward and leg gain scales
            assert np.isnan(res[2, 0]) and np.isnan(res[5, 0])
            rows.append([res[2, 1], res[2, 2], res[5, 1], res[5, 2], res[0, 3], res[0, 4], res[4, 3]])
        out["controllers"].append({"spine_frequency": freq,
                                   "columns": "left wheel velocity, feedforward; right wheel velocity, feedforward; "
                                              "left_hip kp_scale, kd_scale; right_knee kp_scale", "out": rows})
        print("controllers", freq, "final left wheel velocity", rows[-1][0])
    with open(OUT, "w") as f:
        json.dump(out, f)
    print("wrote", OUT, os.path.getsize(OUT) // 1024, "KB")

    # whole observer rows and whole 6 x 6 controller outputs (NaN -> None) of the library on the inputs of
    # test_ref_spine.py::test_reference_library_side_by_side, every SIDE_BY_SIDE_EVERY-th step to keep the file small
    freq, stream = 500, 7
    ref = O.RefSpine(A.default_observer_config(model, float(freq)), A.default_wheel_balancer_config(float(freq)), freq)
    obs_rows = [ref.observers_step(r).tolist() for r in inputs.observer_inputs(A, stream)]
    ctrl_rows = [[None if v != v else v for v in ref.controllers_step(obs3, target, act).reshape(36).tolist()]
                 for obs3, target, act in inputs.controller_inputs(stream)]
    every = SIDE_BY_SIDE_EVERY
    side = {"generator": "tests/golden/make_ref_spine_golden.py", "spine_frequency": freq, "stream": stream,
            "every": every, "observers": obs_rows[::every], "controllers": ctrl_rows[::every]}
    with open(OUT_SIDE, "w") as f:
        json.dump(side, f)
    print("wrote", OUT_SIDE, os.path.getsize(OUT_SIDE) // 1024, "KB")


if __name__ == "__main__":
    main()
