"""Scene reader without MuJoCo (SURVEY 8(f) rank 3): stdlib-XML extraction of what MujocoSimulation.__init__ reads
(mujoco_sim.py:51-91, 258-347).  A small MJCF written here exercises the conversions and the error cases; the
reference's own lab_course.xml, stored as tests/golden/lab_course.xml by make_golden.py, must reproduce the transcribed constants."""
import os
import textwrap

import numpy as np
import pytest

from uav_ac_b200.simulation import scene

MJCF = """
<mujoco model="mini">
  <option timestep="0.002" gravity="0 0 -9.5" integrator="Euler"/>
  <custom>
    <numeric name="planning_bounds" data="0 0 -6 24 14 0"/>
    <numeric name="rotor_force_coefficient" data="1.5"/>
    <numeric name="rotor_drag_to_thrust" data="0.02"/>
    <numeric name="rotor_thrust_limits" data="0.2 5"/>
    <numeric name="motor_time_constants" data="0.01 0.03"/>
    <numeric name="flight_limits" data="3 2 3 12 0.7"/>
  </custom>
  <worldbody>
    <geom name="ground" type="plane" size="1 1 1"/>
    <geom name="obstacle_00" type="box" pos="4 -7 3.1" size="0.3 3 0.3"/>
    <geom name="decor" type="box" pos="1 1 1" size="1 1 1"/>
    <site name="waypoint_01" pos="4 -7 1.3"/>
    <site name="waypoint_00" pos="1 -7 1.3"/>
    <site name="goal" pos="23 -7 2"/>
    <body name="quadrotor" pos="1 -7 0.021">
      <freejoint/>
      <inertial pos="0 0 0" mass="0.6" diaginertia="0.002 0.003 0.004"/>
      <site name="rotor_0" pos="0.12 0.12 0" user="1"/>
      <site name="rotor_1" pos="0.12 -0.12 0" user="-1"/>
      <site name="rotor_2" pos="-0.12 -0.12 0" user="1"/>
      <site name="rotor_3" pos="-0.12 0.12 0" user="-1"/>
    </body>
  </worldbody>
</mujoco>
"""


def _write(tmp_path, text):
    p = tmp_path / "scene.xml"
    p.write_text(textwrap.dedent(text))
    return p


def test_reader_extracts_ned_scene(tmp_path):
    s = scene.load_scene(_write(tmp_path, MJCF))
    assert (s.timestep, s.gravity, s.mass, s.arm_length) == (0.002, 9.5, 0.6, 0.12)
    np.testing.assert_array_equal(s.inertia, [0.002, 0.003, 0.004])
    np.testing.assert_array_equal(s.rotor_spins, [1, -1, 1, -1])
    np.testing.assert_array_equal(s.mission_waypoints, [[1, 7, -0.021], [1, 7, -1.3], [4, 7, -1.3], [23, 7, -2]])   # ENU -> NED, sorted by name
    np.testing.assert_allclose(s.obstacles, [[3.7, 4.3, 4, 10, -3.4, -2.8]])                                        # reference test :246
    np.testing.assert_array_equal(s.goal_position, [23, 7, -2])
    kw = s.quad_kwargs()
    assert kw["force_coefficient"] == 1.5 and kw["drag_to_thrust"] == 0.02 and list(kw["thrust_limits"]) == [0.2, 5.0]
    np.testing.assert_array_equal(s.planning_bounds, [[0, 0, -6], [24, 14, 0]])


@pytest.mark.parametrize("old,new,msg", [
    ('<site name="goal" pos="23 -7 2"/>', "", "missing required element 'goal'"),
    ('name="waypoint_01"', 'name="waypoint_02"', "consecutively numbered"),
    ('type="box" pos="4 -7 3.1"', 'type="sphere" pos="4 -7 3.1"', "must be an axis-aligned box"),
    ('pos="4 -7 3.1" size="0.3 3 0.3"', 'pos="4 -7 3.1" euler="0 0 0.3" size="0.3 3 0.3"', "must be axis-aligned"),
    ('pos="-0.12 0.12 0" user="-1"', 'pos="-0.15 0.12 0" user="-1"', "symmetric X configuration"),
    ('gravity="0 0 -9.5"', 'gravity="0 0 0"', "gravity must be non-zero"),
    ('data="0.2 5"', 'data="0.2"', "must contain 2 values"),
    ('pos="1 -7 0.021"', 'pos="4 -7 3.1"', "start position is inside"),
])
def test_reader_raises_like_the_reference(tmp_path, old, new, msg):
    """ValueError cases of mujoco_sim.py:261-266, 288-291, 317-320, 331-332, 340, 90-91."""
    assert old in MJCF
    with pytest.raises(ValueError, match=msg):
        scene.load_scene(_write(tmp_path, MJCF.replace(old, new)))


def test_lab_course_xml_reproduces_the_transcribed_constants():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lab_course.xml")
    if not os.path.exists(path):
        pytest.skip("tests/golden/lab_course.xml not stored: run tests/golden/make_golden.py with the reference present")
    s = scene.load_scene(path)
    np.testing.assert_allclose(s.mission_waypoints, scene.LAB_COURSE_WAYPOINTS, rtol=0, atol=1e-15)
    np.testing.assert_allclose(s.obstacles, scene.LAB_COURSE_OBSTACLES, rtol=0, atol=1e-12)
    np.testing.assert_array_equal(s.planning_bounds, scene.PLANNING_BOUNDS)
    from oracle import flight_np
    v = flight_np.Vehicle()
    assert (s.timestep, s.gravity, s.mass, s.arm_length, s.force_coefficient, s.drag_to_thrust) == (v.dt, v.g, v.mass, v.arm, v.kf, v.kappa)
    np.testing.assert_array_equal(s.inertia, v.inertia)
    np.testing.assert_array_equal(s.thrust_limits, [v.min_thrust, v.max_thrust])
    np.testing.assert_array_equal(s.motor_time_constants, [v.tau_rise, v.tau_fall])
    np.testing.assert_array_equal(s.flight_limits, [v.max_ascent, v.max_descent, v.max_speed_xy, v.max_horiz_accel, v.max_tilt])
    np.testing.assert_array_equal(s.rotor_spins, [1, -1, 1, -1])


def test_mujoco_to_ned_state_converts_enu_and_flu_frames():
    """tests/unit/simulation/test_mujoco_sim.py:61-74 of the reference, plus a batch."""
    s = scene.mujoco_to_ned_state([1.0, -2.0, 3.0], [np.sqrt(0.5), 0.0, 0.0, np.sqrt(0.5)], [4.0, -5.0, 6.0, 0.1, -0.2, 0.3])
    np.testing.assert_allclose(s, [1, 2, -3, np.sqrt(0.5), 0, 0, -np.sqrt(0.5), 4, 5, -6, 0.1, 0.2, -0.3], rtol=1e-15)
    b = scene.mujoco_to_ned_state(np.zeros((5, 3)), np.tile([2.0, 0, 0, 0], (5, 1)), np.zeros((5, 6)))
    assert b.shape == (5, 13) and np.all(b[:, 3] == 1.0)
    with pytest.raises(ValueError):
        scene.mujoco_to_ned_state([0, 0, 0], [0, 0, 0, 0], np.zeros(6))
    with pytest.raises(ValueError):
        scene.mujoco_to_ned_state([0, 0, np.nan], [1, 0, 0, 0], np.zeros(6))


def test_laboratory_course_is_the_compact_multi_challenge_route():
    """tests/unit/test_utils.py:10-62 of the reference on the transcribed scene and config."""
    from uav_ac_b200 import utils
    cfg, cfg_flight = utils.get_config()
    assert cfg.getint("frequency") > 0 and cfg_flight.getfloat("velocity") > 0 and cfg_flight.getfloat("min_dist_target") == 0.5
    w, obs, lim = scene.LAB_COURSE_WAYPOINTS, scene.LAB_COURSE_OBSTACLES, scene.PLANNING_BOUNDS
    size = lim[1] - lim[0]
    assert size[0] == pytest.approx(24.0) and size[1] == pytest.approx(14.0) and len(w) == 9
    assert np.linalg.norm(np.diff(w, axis=0), axis=1).sum() > 25.0
    lower_alt, upper_alt = -obs[:, 5], -obs[:, 4]                       # NED z is down: altitude = -z
    assert np.any(lower_alt > 2.0) and np.any(np.isclose(lower_alt, 0.0)) and np.any(upper_alt < 3.0)
    assert np.all((w >= lim[0]) & (w <= lim[1]))
    assert np.array_equal(utils.parse_array({"k": "[1, 2, 3]"}, "k"), [1, 2, 3])
