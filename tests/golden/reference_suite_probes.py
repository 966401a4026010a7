# SPDX-License-Identifier: Apache-2.0
"""Probes of the host-side classes whose behaviour the reference's own unit tests specify (tests/utils/ of the
reference: robot state, external force, rotations, point contact). Shared by tests/golden/make_reference_suite_golden.py,
which runs them on the reference's classes, and tests/test_reference_suite_conformance.py, which runs them on
upkie_b200's mirrors aliased under the same module names. Each probe covers the inputs of the matching reference test
file and a few seeded ones, and returns plain JSON values."""
import numpy as np

RANDOMIZATIONS = [
    {"roll": 0.0, "pitch": 0.0},
    {"roll": 0.1, "pitch": 0.2},
    {"roll": 0.05, "pitch": 0.3, "x": 0.1, "z": 0.05, "omega_x": 0.2, "omega_y": 0.4,
     "linear_velocity": [0.5, 0.0, 0.1]},
]


def _state_row(state):
    return (list(np.asarray(state.position_base_in_world, dtype=float)) + _quat(state.orientation_base_in_world)
            + list(np.asarray(state.linear_velocity_base_to_world_in_world, dtype=float))
            + list(np.asarray(state.angular_velocity_base_in_base, dtype=float))
            + list(np.asarray(state.joint_configuration, dtype=float)))


def _quat(rotation):
    """xyzw with a non-negative w: the sign of a quaternion is not part of the rotation."""
    q = np.asarray(rotation.as_quat(), dtype=float)
    return list(-q if q[3] < 0 else q)


def robot_state(modules):
    RobotState = modules["upkie.utils.robot_state"].RobotState
    Randomization = modules["upkie.utils.robot_state_randomization"].RobotStateRandomization
    out = []
    for kw in RANDOMIZATIONS:
        for seed in (0, 1):
            args = {k: np.array(v) if isinstance(v, list) else v for k, v in kw.items()}
            state = RobotState(randomization=Randomization(**args))
            legacy = np.random.RandomState(seed)  # the reference test samples from the np.random module
            out.append({
                "randomization": kw, "seed": seed,
                "orientation_zyx": list(state.sample_orientation(legacy).as_euler("ZYX")),
                "orientation": _quat(state.sample_orientation(np.random.default_rng(seed))),
                "state": _state_row(state.sample_state(np.random.default_rng(seed))),
            })
    return out


def external_force(modules):
    ExternalForce = modules["upkie.utils.external_force"].ExternalForce
    cases = [([1.0, 2.0, 3.0], None), (np.array([4.0, 5.0, 6.0]), True), (np.array([4.0, 5.0, 6.0]), False),
             ([0.0, 0.0, 1.0], None), ([-10.0, -5.0, -1.0], None), ([1000.0, 2000.0, 3000.0], None),
             ([1.123456789, 2.987654321, 3.555555555], None), ([1, 2, 3], True), ([1.0, 2.0], None),
             ([1.0, 2.0, 3.0, 4.0], None), ([], None), (np.array([[1.0, 2.0], [3.0, 4.0]]), None), (5.0, None)]
    out = []
    for force, local in cases:
        try:
            f = ExternalForce(force) if local is None else ExternalForce(force, local=local)
        except ValueError as exc:
            out.append({"error": "ValueError", "message": str(exc)})
            continue
        out.append({"force": f.force.tolist(), "local": f.local, "ndarray": isinstance(f.force, np.ndarray),
                    "dtype": str(f.force.dtype), "repr": repr(f)})
    original = [1.0, 2.0, 3.0]
    f = ExternalForce(original)
    original[0] = 99.0  # the force must not alias the caller's list
    out.append({"after_caller_mutation": f.force.tolist()})
    return out


def rotations(modules):
    rotation_matrix_from_rpy = modules["upkie.utils.rotations"].rotation_matrix_from_rpy
    rng = np.random.default_rng(20261017)
    rpys = [(0.0, 0.0, 0.0), (np.pi, 0.0, 0.0), (0.0, np.pi, 0.0), (0.0, 0.0, np.pi), (np.pi, 0.0, np.pi),
            (0.0, 0.0, np.pi / 2), (0.3, -0.7, 1.2)] + [tuple(rng.uniform(-np.pi, np.pi, 3)) for _ in range(8)]
    return [{"rpy": list(rpy), "R": np.asarray(rotation_matrix_from_rpy(rpy), dtype=float).tolist()} for rpy in rpys]


def point_contact(modules):
    PointContact = modules["upkie.utils.point_contact"].PointContact
    out = []
    for link, pos, force in (("left_wheel_link", [0.1, 0.2, 0.3], [10.0, 20.0, 30.0]),
                             ("imu", [0.0, 0.0, 0.1], [0.0, 0.0, -50.0])):
        c = PointContact(link_name=link, position_contact_in_world=np.array(pos), force_in_world=np.array(force))
        out.append({"link_name": c.link_name, "position": np.asarray(c.position_contact_in_world).tolist(),
                    "force": np.asarray(c.force_in_world).tolist(), "repr": repr(c)})
    return out


# reference test file (relative to its tests/ directory) -> probe
PROBES = {
    "utils/test_robot_state.py": robot_state,
    "utils/test_external_force.py": external_force,
    "utils/test_rotations.py": rotations,
    "utils/test_point_contact.py": point_contact,
}


def mismatches(mine, golden, path="", tol=1e-12):
    """Paths where two probe results differ: numbers beyond ``tol``, anything else not equal."""
    if isinstance(golden, dict):
        if not isinstance(mine, dict) or mine.keys() != golden.keys():
            return [f"{path}: keys {sorted(mine) if isinstance(mine, dict) else mine!r} != {sorted(golden)}"]
        return [m for k in golden for m in mismatches(mine[k], golden[k], f"{path}.{k}", tol)]
    if isinstance(golden, list):
        if not isinstance(mine, list) or len(mine) != len(golden):
            return [f"{path}: {mine!r} != {golden!r}"]
        return [m for k, (a, b) in enumerate(zip(mine, golden)) for m in mismatches(a, b, f"{path}[{k}]", tol)]
    if isinstance(golden, float) and not isinstance(mine, bool) and isinstance(mine, (int, float)):
        return [] if abs(mine - golden) <= tol else [f"{path}: {mine!r} != {golden!r}"]
    return [] if mine == golden else [f"{path}: {mine!r} != {golden!r}"]
