"""The reference's own classes as the CPU arm (oracle/_ref, built by oracle/build_ref.py from a checkout of the reference): the arm
must BE the reference -- it reproduces the committed golden logs and coefficients (made by tests/golden/make_golden.py from the
reference sources) bit for bit -- and the oracle port must agree with it.  The tests of the arm skip where oracle/_ref has not
been built; the oracle is also compared with the reference's outputs stored in tests/golden, which runs everywhere."""
import numpy as np
import pytest

from oracle import flight_np, minsnap_np, ref_arm

needs_arm = pytest.mark.skipif(not ref_arm.available(), reason="oracle/_ref not built (needs a checkout of the reference at build time)")

W = np.array([[1, 7, -0.021], [1, 7, -1.3], [4, 7, -1.3], [7.5, 4, -3], [11, 7, -3.5], [14, 10, -2.5], [17, 10, -3.2], [20.5, 7, -1.4], [23, 7, -2]], dtype=float)
O = np.array([[3.7, 4.3, 4, 10, -3.4, -2.8], [10.7, 11.3, 4, 10, -2.2, 0], [13.3, 14.7, 6.3, 7.7, -6, 0], [20.2, 20.8, 4, 10, -3.3, -2.7]], dtype=float)


@needs_arm
def test_ref_arm_imports_the_byte_compiled_reference_not_the_source_tree():
    import sys
    ns = ref_arm.load()
    assert ns.Quad.__module__ == "uav_ac.quadrotor.quad"
    origin = sys.modules["uav_ac.quadrotor.quad"].__spec__.origin
    assert origin.endswith(".bin") and "oracle/_ref" in origin


@needs_arm
def test_ref_arm_reproduces_the_golden_closed_loop_bit_for_bit(golden):
    gold = golden["closed_loop_v3"]
    tab = ref_arm.mission_table(W, O, 3.0)
    assert tab.shape == (len(gold["X"]), 11)
    n = 2000                                                    # the golden log holds the first 2000 ticks at full rate
    r = ref_arm.fly(tab, W[0], n_ticks=n, obstacles=O, goal=W[-1])
    assert np.array_equal(r["X"], gold["fine"][n - 1, :13]) and np.array_equal(r["omega"], gold["fine"][n - 1, 13:17])
    assert r["periods"] == n // 10 and not r["collision"]


@needs_arm
def test_oracle_port_agrees_with_the_reference_arm_on_a_monte_carlo_vehicle(golden):
    rng = np.random.default_rng(3)
    gs, ms, is_ = rng.uniform(0.8, 1.2, 11), rng.uniform(0.9, 1.1), rng.uniform(0.9, 1.1, 3)
    tab = ref_arm.mission_table(W, O, 3.0)
    r = ref_arm.fly(tab, W[0], n_ticks=1500, gain_scale=gs, mass_scale=ms, inertia_scale=is_, obstacles=O, goal=W[-1])
    veh = flight_np.Vehicle().perturbed(gs, ms, is_)
    p = flight_np.closed_loop(veh, tab, W[0], obstacles=O, goal=W[-1], n_ticks=1500)
    assert np.abs(p["X"] - r["X"]).max() < 1e-9
    # the arm's perturbed-vehicle path is the generator's: the golden Monte-Carlo vehicles' states after 1500 ticks, bit for bit
    var = golden["closed_loop_variants"]
    for j in range(3):
        r = ref_arm.fly(tab, W[0], n_ticks=1500, gain_scale=var[f"mc{j}_gain_scale"], mass_scale=float(var[f"mc{j}_mass_scale"]),
                        inertia_scale=var[f"mc{j}_inertia_scale"], obstacles=O, goal=W[-1])
        assert np.array_equal(r["X"], var[f"mc{j}_X"][1500 // 10 - 1])


def test_oracle_port_agrees_with_the_stored_reference_on_monte_carlo_vehicles(golden):
    """State after 1500 ticks of the golden Monte-Carlo vehicles mc0 and mc2 (mc1 is compared over the whole mission in
    test_oracle_golden.py): the reference's state there is row 149 of its per-period log."""
    tab, var = golden["planning"]["v3_table"], golden["closed_loop_variants"]
    for j in (0, 2):
        veh = flight_np.Vehicle().perturbed(var[f"mc{j}_gain_scale"], float(var[f"mc{j}_mass_scale"]), var[f"mc{j}_inertia_scale"])
        p = flight_np.closed_loop(veh, tab, W[0], obstacles=O, goal=W[-1], n_ticks=1500)
        assert np.abs(p["X"] - var[f"mc{j}_X"][1500 // 10 - 1]).max() < 1e-9


@needs_arm
def test_reference_solver_branches_through_the_arm(golden):
    cs, ts = ref_arm.solve_lstsq(W[1:], 3.0, "solve")
    co, to = minsnap_np.solve_coeffs(W[1:], 3.0, "solve")
    assert np.abs(cs - co).max() / np.abs(cs).max() < 1e-12 and np.allclose(ts, to, rtol=1e-15)
    g = golden["planning"]                                      # the arm is the reference: the stored coefficients, bit for bit
    assert np.array_equal(cs, g["v3_course_coeffs_solve"]) and np.array_equal(ts, g["v3_course_times"])
