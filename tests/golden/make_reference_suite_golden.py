#!/usr/bin/env python
# SPDX-License-Identifier: Apache-2.0
"""Golden results of the reference's own code for tests/test_reference_suite_conformance.py and
tests/test_parity_audit_tool.py, so that those tests compare against the reference on machines without its tree.

Run where the reference tree is present:  python tests/golden/make_reference_suite_golden.py

* ``unit_probes``: tests/golden/reference_suite_probes.py run on the reference's RobotState /
  RobotStateRandomization, ExternalForce, rotation_matrix_from_rpy and PointContact;
* ``backend_suite``: the scenarios of the reference's tests/envs/backends/test_pybullet_backend.py (reset at 0.6 m,
  100 un-actuated steps; the same from a yawed state) run by its own PyBulletBackend on the stand-in ``pybullet``
  whose physics is oracle/ (make_backend_golden.make_fake_pybullet), with and without the joint-limit rows: spine
  observations at the CHECKPOINTS, pitch at every step, and the oracle state the backend's ``_reset_robot_state`` left;
* ``model_suite``: the reference's tests/model/ suite run with its own ``upkie.model`` on the URDFs that
  ``upkie_b200.urdf.write_urdf`` writes (SHA-256 of each file, the suite's verdict, and what its parser reads out);
* ``parity_audit``: tools/parity_audit.py ``record`` of the "torques" scenario on the reference's PyBulletBackend
  (seeds 0 and 1, 40 ticks): the flattened observations of every tick, 10 significant digits.

Output: tests/golden/reference_suite_runs.json.
"""
import hashlib
import importlib.util
import json
import os
import sys
import tempfile
import types
import unittest

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "reference_suite_runs.json")
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

CHECKPOINTS = (0, 1, 2, 5, 10, 20, 50, 100)
BACKEND_STEPS = 100
AUDIT_TICKS = 40


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def _run_suite(mod):
    suite = unittest.defaultTestLoader.loadTestsFromModule(mod)
    result = unittest.TestResult()
    suite.run(result)
    return suite.countTestCases(), [f"{t}: {tb.splitlines()[-1]}" for t, tb in result.failures + result.errors]


def _clear(prefixes):
    for k in [k for k in sys.modules if k.split(".")[0] in prefixes]:
        del sys.modules[k]


def unit_probes():
    import make_wrapper_golden as wg
    import reference_suite_probes as probes

    wg.install_fake_gymnasium()
    wg.load_reference()
    _load("upkie.utils.point_contact", os.path.join(wg.REF, "upkie/utils/point_contact.py"))
    out = {rel: probe(sys.modules) for rel, probe in probes.PROBES.items()}
    _clear(("upkie", "gymnasium", "loop_rate_limiters", "upkie_description"))
    return out


def _reference_backend(urdf, joint_limits):
    import make_backend_golden as bg
    import make_wrapper_golden as wg
    from upkie_b200.model import Model

    wg.install_fake_gymnasium()
    wg.load_reference()
    for name, rel in (("upkie.utils.joystick", "upkie/utils/joystick.py"),
                      ("upkie.utils.point_contact", "upkie/utils/point_contact.py")):
        _load(name, os.path.join(wg.REF, rel))
    sys.modules["upkie_description"].URDF_PATH = urdf
    pb, data = bg.make_fake_pybullet(Model.from_urdf(urdf), urdf, joint_limits=joint_limits)
    sys.modules["pybullet"], sys.modules["pybullet_data"] = pb, data
    backend_mod = _load("upkie.envs.backends.pybullet_backend", os.path.join(wg.REF, "upkie/envs/backends/pybullet_backend.py"))
    return backend_mod, pb


def backend_suite(urdf):
    import make_backend_golden as bg
    import make_wrapper_golden as wg
    from scipy.spatial.transform import Rotation

    out = {}
    for joint_limits in (0, 3):
        backend_mod, pb = _reference_backend(urdf, joint_limits)
        RobotState = sys.modules["upkie.utils.robot_state"].RobotState
        verdict = _run_suite(_load("reference_test_pybullet_backend",
                                   os.path.join(wg.REF, "tests/envs/backends/test_pybullet_backend.py")))
        runs = {}
        for scenario in ("upright", "yawed"):
            backend_mod, pb = _reference_backend(urdf, joint_limits)  # a fresh simulated world per run
            backend = backend_mod.PyBulletBackend(dt=5e-3, gui=False)
            obs = backend.reset(init_state=RobotState(position_base_in_world=np.array([0.0, 0.0, 0.6])))
            run = {"observations": {}, "pitch": []}
            if scenario == "yawed":
                backend._reset_robot_state(RobotState(orientation_base_in_world=Rotation.from_euler("ZYX", [np.pi / 2, 0.0, 0.0])))
                run["state_after_reset_robot_state"] = pb._S.sim.get_state()[0].tolist()
            for t in range(BACKEND_STEPS + 1):
                if t > 0:
                    obs = backend.step(action={})
                    run["pitch"].append(obs["base_orientation"]["pitch"])
                if t in CHECKPOINTS:
                    run["observations"][str(t)] = bg.wg_jsonable(obs)
            backend.close()
            runs[scenario] = run
        out[str(joint_limits)] = {"suite": {"tests": verdict[0], "problems": verdict[1]}, "runs": runs}
        print("backend suite, joint_limits", joint_limits, verdict, "final pitch",
              {s: r["pitch"][-1] for s, r in runs.items()})
        _clear(("upkie", "gymnasium", "pybullet", "pybullet_data", "loop_rate_limiters", "upkie_description"))
    return out


def model_suite():
    import make_wrapper_golden as wg
    from upkie_b200.model import Model
    from upkie_b200.urdf import write_urdf

    ref_root = wg.REF
    tmp = tempfile.mkdtemp()
    upkie_urdf, cookie_urdf = os.path.join(tmp, "upkie.urdf"), os.path.join(tmp, "cookie.urdf")
    write_urdf(Model.standard_upkie(), upkie_urdf, split_fixed_links=True)
    right = Model.standard_upkie()
    right.joint_axis = right.joint_axis.copy()
    right.joint_axis[[2, 5]] *= -1.0
    write_urdf(right, cookie_urdf, split_fixed_links=True)
    for name, path in (("upkie_description", upkie_urdf), ("cookie_description", cookie_urdf)):
        stub = types.ModuleType(name)
        stub.URDF_PATH = path
        sys.modules[name] = stub
    for name, rel in (("upkie", "upkie"), ("upkie.utils", "upkie/utils"), ("upkie.model", "upkie/model")):
        pkg = types.ModuleType(name)
        pkg.__path__ = [os.path.join(ref_root, rel)]
        sys.modules[name] = pkg
    _load("upkie.exceptions", os.path.join(ref_root, "upkie/exceptions.py"))
    for leaf in ("se3", "joint_limit", "joint", "collision_geometry", "link", "kinematic_tree", "model"):
        _load(f"upkie.model.{leaf}", os.path.join(ref_root, f"upkie/model/{leaf}.py"))
    sys.modules["upkie.model"].Model = sys.modules["upkie.model.model"].Model
    total, problems = 0, []
    for rel in ("model/test_model.py", "model/test_kinematic_tree.py", "model/test_se3.py"):
        n, p = _run_suite(_load("reference_test_" + os.path.basename(rel)[:-3], os.path.join(ref_root, "tests", rel)))
        total, problems = total + n, problems + p
    out = {"suite": {"tests": total, "problems": problems}, "urdfs": {}}
    for name, path in (("upkie", upkie_urdf), ("cookie", cookie_urdf)):
        text = open(path, "rb").read()
        m = sys.modules["upkie.model"].Model(path)
        out["urdfs"][name] = {
            "sha256": hashlib.sha256(text).hexdigest(),
            "wheel_radius": m.wheel_radius, "wheel_base": m.wheel_base, "left_wheeled": m.left_wheeled,
            "rotation_base_to_imu": np.asarray(m.rotation_base_to_imu).tolist(),
            "joint_names": [j.name for j in m.joints],
            "upper_leg_joints": [j.name for j in m.upper_leg_joints],
            "wheel_joints": [j.name for j in m.wheel_joints],
        }
    print("model suite", out["suite"])
    _clear(("upkie", "upkie_description", "cookie_description"))
    return out


def parity_audit(urdf):
    import make_wrapper_golden as wg  # noqa: F401

    audit = _load("parity_audit", os.path.join(ROOT, "tools", "parity_audit.py"))
    out = {"ticks": AUDIT_TICKS, "dt": 0.005, "runs": {}}
    for seed in (0, 1):
        backend_mod, pb = _reference_backend(urdf, None)
        RobotState = sys.modules["upkie.utils.robot_state"].RobotState
        ref_model = sys.modules["upkie.model"].Model(urdf)
        tau_max = [float(j.limit.effort) for j in ref_model.joints]
        actions = audit.scenario_actions("torques", AUDIT_TICKS, 0.005, seed, tau_max)
        backend = backend_mod.PyBulletBackend(dt=0.005, model=ref_model)
        header = {"format": "upkie_b200.parity_audit/1", "backend": "pybullet", "scenario": "torques", "seed": 0,
                  "dt": 0.005, "ticks": AUDIT_TICKS, "urdf": "robot.urdf"}
        path = os.path.join(tempfile.mkdtemp(), "run.mpack")
        audit.record(backend, RobotState, actions, header, path)
        backend.close()
        _, records = audit.load(path)
        flats = []
        for rec in records:
            flats.append({})
            audit.flatten("", rec["observation"], flats[-1])
        keys = sorted(flats[0])
        assert all(sorted(f) == keys for f in flats)
        out["runs"][str(seed)] = {"tau_max": tau_max,
                                  "actions_sha256": hashlib.sha256(repr(actions).encode()).hexdigest(),
                                  "keys": keys, "sizes": [len(flats[0][k]) for k in keys],
                                  "observations": [[float(f"{v:.10g}") for k in keys for v in f[k]] for f in flats]}
        _clear(("upkie", "gymnasium", "pybullet", "pybullet_data", "loop_rate_limiters", "upkie_description"))
    return out


def main():
    from upkie_b200.model import Model
    from upkie_b200.urdf import write_urdf

    urdf = os.path.join(tempfile.mkdtemp(), "robot.urdf")
    write_urdf(Model.standard_upkie(), urdf, split_fixed_links=False)
    out = {"generator": "tests/golden/make_reference_suite_golden.py", "probes": "tests/golden/reference_suite_probes.py",
           "unit_probes": unit_probes(), "backend_suite": backend_suite(urdf), "model_suite": model_suite(),
           "parity_audit": parity_audit(urdf)}
    with open(OUT, "w") as f:
        json.dump(out, f)
    print("wrote", OUT, os.path.getsize(OUT) // 1024, "KB")


if __name__ == "__main__":
    main()
