# SPDX-License-Identifier: Apache-2.0
"""tools/parity_audit.py: the record / compare logic, exercised on the reference's own ``PyBulletBackend`` (loaded
unmodified from the reference tree, ``pybullet`` replaced by the stand-in whose physics is oracle/), and on that
backend's observations as recorded in tests/golden/reference_suite_runs.json where the tree is absent. The tool's
purpose - a run against a REAL PyBullet - needs a machine that has one."""
import importlib.util
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("UPKIE_REFERENCE", "/root/reference")


@pytest.fixture()
def audit():
    spec = importlib.util.spec_from_file_location("parity_audit", os.path.join(ROOT, "tools", "parity_audit.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_scenarios_are_open_loop_and_seeded(audit):
    tau_max = [16.0, 16.0, 1.7, 16.0, 16.0, 1.7]
    for name in audit.SCENARIOS:
        a = audit.scenario_actions(name, 50, 0.005, 3, tau_max)
        b = audit.scenario_actions(name, 50, 0.005, 3, tau_max)
        assert repr(a) == repr(b)  # same seed, same actions (NaN positions included)
        if name == "fall":
            assert a == [{}] * 50  # no action: the robot topples onto its collision shapes
            continue
        assert len(a) == 50 and set(a[0]["servo"]) == set(audit.JOINTS)
        for joint, servo in a[7]["servo"].items():
            assert abs(servo["feedforward_torque"]) <= servo["maximum_torque"] and not np.isnan(servo["velocity"])
    assert repr(audit.scenario_actions("torques", 5, 0.005, 1, tau_max)) != repr(
        audit.scenario_actions("torques", 5, 0.005, 2, tau_max))


def _check_recordings(audit, paths, ticks):
    """Three "torques" recordings: seeds 0, 0 and 1."""
    header, records = audit.load(paths[0])
    assert header["scenario"] == "torques" and len(records) == ticks + 1
    assert records[0]["tick"] == 0 and records[-1]["tick"] == ticks
    assert set(records[1]["action"]["servo"]) == set(audit.JOINTS)
    same = audit.compare(paths[0], paths[1])
    assert "servo.left_knee.position" in same and "imu.orientation" in same
    assert max(max(row.values()) for row in same.values()) == 0.0  # same inputs, same backend: identical
    other = audit.compare(paths[0], paths[2])  # different torques: the table shows it
    assert other["servo.left_knee.velocity"][ticks] > 1e-2
    assert sorted(other["servo.left_knee.velocity"]) == [1, 2, 5, 10, 20, 40]
    audit.print_table(other)


class _ReplayBackend:
    """Serves, tick by tick, the observations the reference's PyBulletBackend returned for the same actions
    (tests/golden/make_reference_suite_golden.py)."""

    def __init__(self, run):
        self._keys, self._sizes, self._rows = run["keys"], run["sizes"], run["observations"]
        self._k = 0

    def _observation(self):
        row, out, i = self._rows[self._k], {}, 0
        for key, size in zip(self._keys, self._sizes):
            out[key] = row[i:i + size]
            i += size
        self._k += 1
        return out

    def reset(self, init_state):
        self._k = 0
        return self._observation()

    def step(self, action):
        return self._observation()


def _record_and_compare_recorded_runs(audit, tmp_path):
    import hashlib
    import json

    with open(os.path.join(os.path.dirname(__file__), "golden", "reference_suite_runs.json")) as f:
        golden = json.load(f)["parity_audit"]
    from upkie_b200.robot_state import RobotState

    dt, ticks = golden["dt"], golden["ticks"]
    paths = []
    for run, scenario_seed in enumerate((0, 0, 1)):
        recorded = golden["runs"][str(scenario_seed)]
        actions = audit.scenario_actions("torques", ticks, dt, scenario_seed, recorded["tau_max"])
        assert hashlib.sha256(repr(actions).encode()).hexdigest() == recorded["actions_sha256"]  # what the reference saw
        header = {"format": "upkie_b200.parity_audit/1", "backend": "pybullet", "scenario": "torques",
                  "seed": 0, "dt": dt, "ticks": ticks, "urdf": "robot.urdf"}
        path = str(tmp_path / f"recorded{run}.mpack")
        audit.record(_ReplayBackend(recorded), RobotState, actions, header, path)
        paths.append(path)
    _check_recordings(audit, paths, ticks)


def test_record_and_compare_on_the_reference_backend(audit, tmp_path):
    """On the reference backend's recorded observations everywhere, and on the backend itself where the reference
    tree is present."""
    _record_and_compare_recorded_runs(audit, tmp_path)
    if not os.path.exists(os.path.join(REF, "upkie", "envs", "backends", "pybullet_backend.py")):
        return
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import make_backend_golden as bg
    import make_wrapper_golden as wg
    from upkie_b200.model import Model
    from upkie_b200.urdf import write_urdf

    names = ("upkie", "gymnasium", "pybullet", "pybullet_data", "loop_rate_limiters", "upkie_description")
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] in names}
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
        spec = importlib.util.spec_from_file_location(
            "upkie.envs.backends.pybullet_backend", os.path.join(wg.REF, "upkie/envs/backends/pybullet_backend.py"))
        backend_mod = importlib.util.module_from_spec(spec)
        sys.modules["upkie.envs.backends.pybullet_backend"] = backend_mod
        pb, data = bg.make_fake_pybullet(Model.from_urdf(urdf), urdf)
        sys.modules["pybullet"], sys.modules["pybullet_data"] = pb, data
        spec.loader.exec_module(backend_mod)
        robot_state_cls = sys.modules["upkie.utils.robot_state"].RobotState
        ref_model = sys.modules["upkie.model"].Model(urdf)
        tau_max = [float(j.limit.effort) for j in ref_model.joints]
        dt, ticks = 0.005, 40
        paths = []
        for run, scenario_seed in enumerate((0, 0, 1)):
            pb, data = bg.make_fake_pybullet(Model.from_urdf(urdf), urdf)  # a fresh simulated world per run
            sys.modules["pybullet"], sys.modules["pybullet_data"] = pb, data
            backend_mod.pybullet, backend_mod.pybullet_data = pb, data
            backend = backend_mod.PyBulletBackend(dt=dt, model=ref_model)
            actions = audit.scenario_actions("torques", ticks, dt, scenario_seed, tau_max)
            header = {"format": "upkie_b200.parity_audit/1", "backend": "pybullet", "scenario": "torques",
                      "seed": 0, "dt": dt, "ticks": ticks, "urdf": urdf}
            path = str(tmp_path / f"run{run}.mpack")
            audit.record(backend, robot_state_cls, actions, header, path)
            backend.close()
            paths.append(path)
        _check_recordings(audit, paths, ticks)
    finally:
        for k in [k for k in sys.modules if k.split(".")[0] in names]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_constants_report_flags_differences(audit):
    """`parity_audit.py constants`: the report logic on a made-up PyBullet answer (a real one needs a machine that has
    pybullet): every restated Bullet constant of UpkieSimConfig is looked up under its PyBullet name."""
    from upkie_b200 import _abi

    cfg = _abi.default_sim_config()
    physics = {"numSolverIterations": 50, "solverResidualThreshold": 1e-7, "contactBreakingThreshold": 0.02,
               "contactERP": 0.2, "erp": 0.2}
    dynamics = {"left_wheel_tire": {"contactStiffness": 30000.0, "contactDamping": 1000.0, "lateralFriction": 1.0},
                "torso": {"lateralFriction": 0.5}, "": {"linearDamping": 0.04, "angularDamping": 0.04}}
    rows = {field: (ours, key, theirs) for field, ours, key, theirs in audit.constants_report(cfg, physics, dynamics)}
    assert rows["solver_residual_threshold"] == (1e-7, "solverResidualThreshold", 1e-7)
    assert rows["pgs_iterations"][2] == 50.0 and rows["contact_stiffness"][2] == 30000.0
    assert rows["warmstarting_factor"][2] is None  # a key this PyBullet did not report
    assert all(theirs is None or abs(theirs - ours) < 1e-9 for ours, _, theirs in rows.values())
    for field, _, _ in audit.RESTATED_CONSTANTS:
        assert hasattr(cfg, field)
