# SPDX-License-Identifier: Apache-2.0
"""Runs the REFERENCE'S OWN unit tests against this package's mirrors of the reference's host-side types.

Where the reference tree is present, its test files for the types we mirror are loaded as they are and executed with
``upkie.utils.robot_state`` / ``robot_state_randomization`` / ``external_force`` aliased to ``upkie_b200``'s classes:
a user switching packages keeps the behaviour those tests specify. Everywhere, the same comparisons run against what
the reference's code produced when tests/golden/make_reference_suite_golden.py ran it (reference_suite_runs.json)."""
import hashlib
import importlib.util
import json
import os
import sys
import types
import unittest

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import reference_suite_probes as probes  # noqa: E402

REF_TESTS = os.path.join(os.environ.get("UPKIE_REFERENCE", "/root/reference"), "tests")

CASES = [
    ("utils/test_robot_state.py", "robot state and its randomisation"),
    ("utils/test_external_force.py", "ExternalForce validation"),
    ("utils/test_rotations.py", "rotation_matrix_from_rpy of the URDF loader"),
    ("utils/test_point_contact.py", "PointContact of Backend.get_contact_points"),
]


@pytest.fixture(scope="module")
def golden():
    with open(os.path.join(os.path.dirname(__file__), "golden", "reference_suite_runs.json")) as f:
        return json.load(f)


@pytest.fixture()
def aliased_upkie():
    import upkie_b200.model as b200_model
    import upkie_b200.robot_state as b200_state

    saved = {k: v for k, v in sys.modules.items() if k == "upkie" or k.startswith("upkie.")}
    for k in saved:
        del sys.modules[k]
    pkg = types.ModuleType("upkie")
    pkg.__path__ = []
    utils = types.ModuleType("upkie.utils")
    utils.__path__ = []
    rs = types.ModuleType("upkie.utils.robot_state")
    rs.RobotState = b200_state.RobotState
    rsr = types.ModuleType("upkie.utils.robot_state_randomization")
    rsr.RobotStateRandomization = b200_state.RobotStateRandomization
    ef = types.ModuleType("upkie.utils.external_force")
    ef.ExternalForce = b200_model.ExternalForce
    import upkie_b200.urdf as b200_urdf

    rot = types.ModuleType("upkie.utils.rotations")
    rot.rotation_matrix_from_rpy = b200_urdf.rotation_matrix_from_rpy
    pc = types.ModuleType("upkie.utils.point_contact")
    pc.PointContact = b200_model.PointContact
    sys.modules.update({"upkie": pkg, "upkie.utils": utils, "upkie.utils.robot_state": rs,
                        "upkie.utils.robot_state_randomization": rsr, "upkie.utils.external_force": ef,
                        "upkie.utils.rotations": rot, "upkie.utils.point_contact": pc})
    try:
        yield
    finally:
        for k in [k for k in sys.modules if k == "upkie" or k.startswith("upkie.")]:
            del sys.modules[k]
        sys.modules.update(saved)


@pytest.mark.parametrize("rel,what", CASES)
def test_reference_unit_tests_pass_on_our_mirrors(aliased_upkie, golden, rel, what):
    """The probes of tests/golden/reference_suite_probes.py (the inputs of the reference's test file and a few seeded
    ones) give on our mirrors what they gave on the reference's classes; the test file itself where it is present."""
    problems = probes.mismatches(probes.PROBES[rel](sys.modules), golden["unit_probes"][rel])
    assert not problems, f"{what}: {problems[:5]}"
    path = os.path.join(REF_TESTS, rel)
    if not os.path.exists(path):
        return
    spec = importlib.util.spec_from_file_location("reference_test_" + os.path.basename(rel)[:-3], path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    suite = unittest.defaultTestLoader.loadTestsFromModule(mod)
    assert suite.countTestCases() > 0
    result = unittest.TestResult()
    suite.run(result)
    problems = [f"{t}: {tb.splitlines()[-1]}" for t, tb in result.failures + result.errors]
    assert not problems, f"{what}: {problems}"


def _replay_backend_suite(golden, joint_limits, tmp_path, oracle_lib):
    """The runs behind the reference's backend suite, recorded from its PyBulletBackend on the stand-in whose physics
    is oracle/, replayed by the oracle's restatement of that backend: every step's pitch and the whole spine
    observation at the recorded checkpoints."""
    from test_backend_golden import _action, _compare, _row64
    from upkie_b200 import _abi as A
    from upkie_b200.model import Model
    from upkie_b200.urdf import write_urdf

    g = golden["backend_suite"][str(joint_limits)]
    assert g["suite"]["tests"] >= 4
    assert not [p for p in g["suite"]["problems"] if not (joint_limits and "test_fall_pitch" in p)], g["suite"]
    urdf = str(tmp_path / "robot.urdf")
    write_urdf(Model.standard_upkie(), urdf, split_fixed_links=False)
    model = Model.from_urdf(urdf)
    upright = np.zeros(A.INIT_DIM)
    upright[2], upright[3] = 0.6, 1.0  # RobotState(position_base_in_world=[0, 0, 0.6]) of the suite's setUp
    action, absent = _action([None] * 6)  # step(action={}): no joint commanded
    for scenario, run in g["runs"].items():
        cfg = A.default_sim_config()
        cfg.joint_limits = joint_limits
        osim = oracle_lib.OracleSim(model, cfg, 1, threads=1)
        osim.reset(upright.reshape(1, -1))
        if scenario == "yawed":  # backend._reset_robot_state(yaw = pi / 2) after setUp's reset
            osim.set_state(np.asarray(run["state_after_reset_robot_state"]).reshape(1, -1))
        for t in range(len(run["pitch"]) + 1):
            if t > 0:
                osim.step_servos(action.reshape(1, 6, 6))
                assert abs(osim.spine_obs()[0][A.SP_PITCH] - run["pitch"][t - 1]) < 1e-9, (scenario, t)
            if str(t) not in run["observations"]:
                continue
            mine, ref = osim.spine_obs()[0], _row64(run["observations"][str(t)])
            if scenario == "yawed" and t == 1:
                # the backend's IMU finite difference spans its _reset_robot_state, which set_state does not carry
                for block in (A.SP_IMU_LINACC, A.SP_IMU_RAWACC):
                    mine[block:block + 3] = ref[block:block + 3]
            _compare(mine, ref, 1e-8, skip_torque=absent)
        assert abs(run["pitch"][0]) < 1e-7  # the suite's pitch right after the reset
        if not joint_limits:
            assert abs(run["pitch"][-1]) > 0.5  # and the fall within 100 steps


@pytest.mark.parametrize("joint_limits", [0, 3])
def test_reference_pybullet_backend_suite_passes_on_our_physics(tmp_path, golden, oracle_lib, joint_limits):
    """tests/envs/backends/test_pybullet_backend.py of the reference (its tests of the REAL PyBullet backend: step
    returns a dict, pitch 0 after a step, the robot falls within 100 un-actuated steps, also from a yawed start)
    executed unmodified with ``pybullet`` replaced by the stand-in whose physics is oracle/ and ``upkie_description``
    pointing at a URDF written by upkie_b200: what the reference expects of Bullet at that level holds for the
    restated physics. With the joint-limit rows on (the default since round 2) the two "fallen at step 100" samples
    depend on the stand-in inertias (tests/test_oracle_pins.py::test_pitch_zero_after_one_step_and_fall_without_action);
    they are the only tests allowed to deviate, and the oracle pins assert the fall itself. The suite's runs as
    recorded from the reference (tests/golden/reference_suite_runs.json) are replayed everywhere; the suite itself
    runs where the reference tree is present."""
    _replay_backend_suite(golden, joint_limits, tmp_path, oracle_lib)
    path = os.path.join(REF_TESTS, "envs", "backends", "test_pybullet_backend.py")
    if not os.path.exists(path):
        return
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import make_backend_golden as bg
    import make_wrapper_golden as wg
    from upkie_b200.model import Model
    from upkie_b200.urdf import write_urdf

    saved = {k: v for k, v in sys.modules.items()
             if k.split(".")[0] in ("upkie", "gymnasium", "pybullet", "pybullet_data", "loop_rate_limiters", "upkie_description")}
    try:
        wg.install_fake_gymnasium()
        wg.load_reference()
        for name, rel in (("upkie.utils.joystick", "upkie/utils/joystick.py"),
                          ("upkie.utils.point_contact", "upkie/utils/point_contact.py")):
            spec = importlib.util.spec_from_file_location(name, os.path.join(wg.REF, rel))
            mod = importlib.util.module_from_spec(spec)
            sys.modules[name] = mod
            spec.loader.exec_module(mod)
        urdf = str(tmp_path / "robot.urdf")
        write_urdf(Model.standard_upkie(), urdf, split_fixed_links=False)
        sys.modules["upkie_description"].URDF_PATH = urdf
        pb, data = bg.make_fake_pybullet(Model.from_urdf(urdf), urdf, joint_limits=joint_limits)
        sys.modules["pybullet"], sys.modules["pybullet_data"] = pb, data
        spec = importlib.util.spec_from_file_location(
            "upkie.envs.backends.pybullet_backend", os.path.join(wg.REF, "upkie/envs/backends/pybullet_backend.py"))
        backend_mod = importlib.util.module_from_spec(spec)
        sys.modules["upkie.envs.backends.pybullet_backend"] = backend_mod
        spec.loader.exec_module(backend_mod)
        spec = importlib.util.spec_from_file_location("reference_test_pybullet_backend", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        suite = unittest.defaultTestLoader.loadTestsFromModule(mod)
        assert suite.countTestCases() >= 4
        result = unittest.TestResult()
        suite.run(result)
        problems = [f"{t}: {tb.splitlines()[-1]}" for t, tb in result.failures + result.errors]
        if joint_limits:
            problems = [p for p in problems if "test_fall_pitch" not in p]
        assert not problems, problems
    finally:
        for k in [k for k in sys.modules
                  if k.split(".")[0] in ("upkie", "gymnasium", "pybullet", "pybullet_data", "loop_rate_limiters", "upkie_description")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_reference_model_suite_passes_on_urdfs_written_by_upkie_b200(tmp_path, golden):
    """tests/model/test_model.py, test_kinematic_tree.py and test_se3.py of the reference, unmodified, run with the
    reference's OWN ``upkie.model`` package while ``upkie_description.URDF_PATH`` / ``cookie_description.URDF_PATH``
    point at URDFs written by ``upkie_b200.urdf.write_urdf`` (left- and right-wheeled stand-ins): wheel radius 0.05,
    wheel base 0.3048, base -> IMU rotation, torso at (0, 0, -0.1), frame names, tire cylinders, left / right
    wheeledness - every constant the reference pins on its model comes out of our file through its parser.
    Everywhere: the files written now are byte for byte those on which the suite passed when
    tests/golden/make_reference_suite_golden.py ran it, and our loader reads out of them what the reference's parser
    read; the suite itself runs where the reference tree is present."""
    from upkie_b200.model import Model
    from upkie_b200.urdf import write_urdf

    upkie_urdf, cookie_urdf = str(tmp_path / "upkie.urdf"), str(tmp_path / "cookie.urdf")
    write_urdf(Model.standard_upkie(), upkie_urdf, split_fixed_links=True)
    right = Model.standard_upkie()
    right.joint_axis = right.joint_axis.copy()
    right.joint_axis[[2, 5]] *= -1.0  # wheel axes reversed: a right-wheeled (Cookie-style) robot
    write_urdf(right, cookie_urdf, split_fixed_links=True)
    g = golden["model_suite"]
    assert g["suite"]["tests"] >= 30 and not g["suite"]["problems"], g["suite"]
    for name, path in (("upkie", upkie_urdf), ("cookie", cookie_urdf)):
        ref = g["urdfs"][name]
        with open(path, "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == ref["sha256"], name
        m = Model.from_urdf(path)
        assert m.wheel_radius == pytest.approx(ref["wheel_radius"], abs=1e-12)
        assert m.wheel_base == pytest.approx(ref["wheel_base"], abs=1e-12)
        assert m.left_wheeled == ref["left_wheeled"]
        assert np.allclose(m.rotation_base_to_imu, np.asarray(ref["rotation_base_to_imu"]), atol=1e-12)
        assert [j.name for j in m.joints] == ref["joint_names"]
        assert [j.name for j in m.upper_leg_joints] == ref["upper_leg_joints"]
        assert [j.name for j in m.wheel_joints] == ref["wheel_joints"]
    if not os.path.exists(os.path.join(REF_TESTS, "model", "test_model.py")):
        return

    ref_root = os.path.dirname(REF_TESTS)
    saved = {k: v for k, v in sys.modules.items()
             if k.split(".")[0] in ("upkie", "upkie_description", "cookie_description")}
    for k in saved:
        del sys.modules[k]
    try:
        for name, path in (("upkie_description", upkie_urdf), ("cookie_description", cookie_urdf)):
            stub = types.ModuleType(name)
            stub.URDF_PATH = path
            sys.modules[name] = stub
        pkg = types.ModuleType("upkie")
        pkg.__path__ = [os.path.join(ref_root, "upkie")]
        sys.modules["upkie"] = pkg

        def load(name, rel):
            spec = importlib.util.spec_from_file_location(name, os.path.join(ref_root, rel))
            mod = importlib.util.module_from_spec(spec)
            sys.modules[name] = mod
            spec.loader.exec_module(mod)
            return mod

        load("upkie.exceptions", "upkie/exceptions.py")
        utils = types.ModuleType("upkie.utils")
        utils.__path__ = [os.path.join(ref_root, "upkie", "utils")]
        sys.modules["upkie.utils"] = utils
        model_pkg = types.ModuleType("upkie.model")
        model_pkg.__path__ = [os.path.join(ref_root, "upkie", "model")]
        sys.modules["upkie.model"] = model_pkg
        for leaf in ("se3", "joint_limit", "joint", "collision_geometry", "link", "kinematic_tree", "model"):
            load(f"upkie.model.{leaf}", f"upkie/model/{leaf}.py")
        model_pkg.Model = sys.modules["upkie.model.model"].Model
        total = 0
        for rel in ("model/test_model.py", "model/test_kinematic_tree.py", "model/test_se3.py"):
            mod = load("reference_test_" + os.path.basename(rel)[:-3], os.path.join("tests", rel))
            suite = unittest.defaultTestLoader.loadTestsFromModule(mod)
            total += suite.countTestCases()
            result = unittest.TestResult()
            suite.run(result)
            problems = [f"{t}: {tb.splitlines()[-1]}" for t, tb in result.failures + result.errors]
            assert not problems, (rel, problems)
        assert total >= 30
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] in ("upkie", "upkie_description", "cookie_description")]:
            del sys.modules[k]
        sys.modules.update(saved)
