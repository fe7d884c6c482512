"""Configurations the one-engine-per-test parity suites never reach, each tick against the C oracle fed the exported Philox
noise: several live handles of one kernel instantiation with different horizons (the shared-memory opt-in is per function,
not per handle), a fleet with one robot's state NaN, the two-level merge per robot, batched obstacle and cost-mode kernels,
one CTA per robot, the boundaries where a handle switches rollout path (regenerate / noise stash / time-parallel), and the
two drop-in classes no other test runs on the GPU."""
import os
import re
import threading

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from golden_util import Golden  # noqa: E402
from gpu_util import engine_from_spec  # noqa: E402
from oracle import c_oracle as co  # noqa: E402
from oracle import mppi_oracle as orc  # noqa: E402

U_ATOL_DD = 2e-5        # updated nominal, diff-drive (test_gpu_parity.py)
U_ATOL_RC = 1e-4        # race-car: FP32 class, controls of O(1) (test_gpu_tpar.py, test_gpu_fullsize.py)
MPPI_E_NUMERIC = -7


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def _f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


def _dd_spec(K, T, obstacles=None, cost_mode="sum"):
    sp = orc.diffdrive_spec(K=K, T=T, param_exploration=0.05, cost_mode=cost_mode, waypoint_mode="frozen",
                            obstacles=obstacles, margin=1.0 if obstacles is None else 1.2)
    sp.temperature = 2.0
    return sp


def _rc_case(K, T):
    """Race-car class with its obstacles (mppi_race_car_obstacle.py), dynamic 200-entry window."""
    g = Golden("racecar_alpha0.9")
    sp = g.spec()
    sp.K, sp.T = K, T
    return sp, g.path, np.asarray(g.rec["x0"][0], dtype=np.float64)


def _dd_case(K, T):
    return _dd_spec(K, T), Golden("diffdrive_pe0.05").path, np.array([0.3, 0.2, 0.4])


def _create(sp, path, capfd):
    """Engine plus the rollout path and grid mppi_create selected (printed when MPPI_VERBOSE is set)."""
    capfd.readouterr()
    old = os.environ.get("MPPI_VERBOSE")
    os.environ["MPPI_VERBOSE"] = "1"
    try:
        eng = engine_from_spec(sp, path)
    finally:
        if old is None:
            del os.environ["MPPI_VERBOSE"]
        else:
            os.environ["MPPI_VERBOSE"] = old
    sel = re.findall(r"rollout path (\w+), (\d+) CTAs per robot", capfd.readouterr().err)
    assert len(sel) == 1, sel
    return eng, sel[0][0], int(sel[0][1])


def _oracle_tick(eng, sp, path, U, idx, x0, seed, tick, robot=0):
    eps = torch.zeros(sp.K, sp.T, 2, dtype=torch.float32, device="cuda")
    eng.generate_noise(eps, seed=seed, tick=tick, robot=robot)
    return co.tick(sp, path, U, int(idx), _f32(x0), eps.cpu().numpy())


class _Handle:
    """One single-robot handle; every Philox tick is checked against the oracle and carries the nominal forward."""

    def __init__(self, sp, path, x0, tol):
        self.sp, self.path, self.x0, self.tol = sp, path, x0, tol
        self.eng = engine_from_spec(sp, path)
        self.U, self.idx, self.tick = np.zeros((sp.T, 2)), 0, 0

    def step_and_check(self):
        u0, useq = self.eng.step(self.x0, None, seed=17, tick=self.tick)
        u0, useq = u0.copy(), useq.copy()
        idx = self.eng.get_waypoint_idx()
        o = _oracle_tick(self.eng, self.sp, self.path, self.U, self.idx, self.x0, 17, self.tick)
        where = (self.sp.T, self.tick)
        assert np.max(np.abs(useq - o["U_after"])) <= self.tol, (where, np.max(np.abs(useq - o["U_after"])))
        assert np.max(np.abs(u0 - o["u0"])) <= self.tol, where
        assert idx == o["idx_after"], where
        self.U, self.idx, self.tick = useq.astype(np.float64), idx, self.tick + 1


# ---- A. two live handles of the same instantiation, different horizons ------------------------------------------------
# diff-drive static window with the noise stash: T = 50 needs 100 KB of dynamic shared memory, T = 30 60 KB; race-car
# time-parallel rollout: T = 50 77 KB, T = 25 38 KB.  Creating the second handle must not lower the first one's opt-in.
PAIRS = {"diffdrive_stash": (lambda T: _dd_case(4096, T), (50, 30), "stash", U_ATOL_DD),
         "racecar_tpar": (lambda T: _rc_case(16384, T), (50, 25), "tpar", U_ATOL_RC)}


@pytest.mark.parametrize("kind,order,threaded", [("diffdrive_stash", "large_first", False),
                                                 ("diffdrive_stash", "small_first", False),
                                                 ("racecar_tpar", "large_first", False),
                                                 ("racecar_tpar", "small_first", False),
                                                 ("diffdrive_stash", "large_first", True)])
def test_coexisting_handles_with_different_horizons_both_tick_correctly(kind, order, threaded, capfd):
    case, (t_large, t_small), want_path, tol = PAIRS[kind]
    t_first, t_second = (t_large, t_small) if order == "large_first" else (t_small, t_large)
    first = _Handle(*case(t_first), tol)
    first.step_and_check()
    if threaded:
        made, failed = [], []

        def make():
            try:
                made.append(_Handle(*case(t_second), tol))
            except Exception as e:                  # noqa: BLE001 -- re-raised in the test's thread
                failed.append(e)
        th = threading.Thread(target=make)
        th.start()
        th.join()
        if failed:
            raise failed[0]
        second = made[0]
    else:
        second = _Handle(*case(t_second), tol)
    first.step_and_check()
    second.step_and_check()
    first.eng.close()
    second.eng.close()
    for T in (t_first, t_second):                   # both horizons really took the path whose opt-in is shared
        sp, path, _ = case(T)
        eng, sel, _ = _create(sp, path, capfd)
        eng.close()
        assert sel == want_path, (kind, T, sel)


# ---- B. a non-finite state in a fleet -----------------------------------------------------------------------------------
BAD = 3


def _fleet_states(path, R, seed):
    rng = np.random.default_rng(seed)
    return np.stack([np.append(path[(7 * r) % 140, :2] + rng.normal(0, 0.1, 2), path[(7 * r) % 140, 2] + rng.normal(0, 0.1))
                     for r in range(R)])


@pytest.mark.parametrize("R", [6, 300])            # several CTAs per robot (ticket merge) / one CTA per robot
def test_fleet_nan_state_fails_only_that_robot_and_is_reported(R):
    from mppi_b200 import MppiError
    from mppi_b200.batched import BatchedMPPI
    K, T = 1024, 30
    path = Golden("diffdrive_pe0.05").path
    x0 = _fleet_states(path, R, 21)
    x_bad = x0.copy()
    x_bad[BAD] = np.nan
    others = np.arange(R) != BAD

    def fleet():
        return BatchedMPPI(R, path, num_samples_K=K, num_horizons_T=T, temperature=2.0, seed=13)

    ref = fleet()                                   # the same fleet with every state finite
    ref_ticks = []
    for _ in range(2):
        u0 = ref.step(_dev(x0)).clone()
        ref_ticks.append((u0.cpu().numpy(), ref.nominal(), ref.waypoint_idx()))
    ref.engine.close()

    b = fleet()
    U_init, i_init = b.nominal(), b.waypoint_idx()
    u0 = b.step(_dev(x_bad)).clone()
    with pytest.raises(MppiError, match="robot %d:" % BAD):
        b.engine.synchronize()
    u0 = u0.cpu().numpy()
    Un, iN = b.nominal(), b.waypoint_idx()          # the fault was reported once: no second error
    assert np.all(np.isnan(u0[BAD])), u0[BAD]
    assert np.array_equal(Un[BAD], U_init[BAD]) and iN[BAD] == i_init[BAD]
    # robots own their CTAs and Philox streams: the others are bit-identical to the all-finite fleet
    assert np.array_equal(u0[others], ref_ticks[0][0][others])
    assert np.array_equal(Un[others], ref_ticks[0][1][others]) and np.array_equal(iN[others], ref_ticks[0][2][others])

    # the next tick, every state finite, is judged on its own
    u1 = b.step(_dev(x0)).clone()
    b.engine.synchronize()
    u1 = u1.cpu().numpy()
    U1, i1 = b.nominal(), b.waypoint_idx()
    assert np.array_equal(u1[others], ref_ticks[1][0][others]) and np.array_equal(U1[others], ref_ticks[1][1][others])
    assert np.array_equal(i1[others], ref_ticks[1][2][others])
    sp = _dd_spec(K, T)
    o = _oracle_tick(b.engine, sp, path, U_init[BAD].astype(np.float64), i_init[BAD], x0[BAD], 13, 1, robot=BAD)
    assert np.max(np.abs(U1[BAD] - o["U_after"])) <= U_ATOL_DD, np.max(np.abs(U1[BAD] - o["U_after"]))
    assert np.max(np.abs(u1[BAD] - o["u0"])) <= U_ATOL_DD and i1[BAD] == o["idx_after"]
    b.engine.close()


def test_fleet_closed_loop_nan_state_is_reported_and_only_that_robot_logs_nan():
    from mppi_b200 import _lib
    from mppi_b200.batched import BatchedMPPI
    R, K, T, n = 6, 1024, 20, 8
    path = Golden("diffdrive_pe0.05").path
    x0 = _fleet_states(path, R, 22)
    x_bad = x0.copy()
    x_bad[BAD] = np.nan

    def run(x):
        # through the C ABI: the Python wrapper raises on MPPI_E_NUMERIC and would drop the logs
        b = BatchedMPPI(R, path, num_samples_K=K, num_horizons_T=T, temperature=2.0, seed=13)
        eng = b.engine
        xs = np.ascontiguousarray(x, dtype=np.float64)
        states = np.zeros((n + 1, R, 3), dtype=np.float32)
        controls = np.zeros((n, R, 2), dtype=np.float32)
        st = eng.lib.mppi_run_closed_loop(eng._h, xs.ctypes.data_as(_lib._PD), n, b.seed, 0, 0,
                                          states.ctypes.data_as(_lib._PF), controls.ctypes.data_as(_lib._PF))
        err = eng.lib.mppi_last_error(eng._h).decode()
        again = eng.lib.mppi_synchronize(eng._h)
        eng.close()
        return st, err, again, states, controls

    st, _, _, states_ok, controls_ok = run(x0)
    assert st == 0 and np.all(np.isfinite(states_ok)) and np.all(np.isfinite(controls_ok))
    st, err, again, states, controls = run(x_bad)
    assert st == MPPI_E_NUMERIC and ("robot %d:" % BAD) in err, (st, err)
    assert again == 0                                   # reported once, then cleared
    assert np.all(np.isnan(states[1:, BAD])) and np.all(np.isnan(controls[:, BAD]))
    others = np.arange(R) != BAD
    assert np.array_equal(states[:, others], states_ok[:, others])
    assert np.array_equal(controls[:, others], controls_ok[:, others])


# ---- C. fleets against the oracle: two-level merge per robot, obstacle / cost-mode kernels, one CTA per robot ------------
def _fleet_vs_oracle(b, sp, path, x0, robots, tol, ticks=2):
    """Steps the fleet `ticks` times from zero nominals; robots in `robots` are checked against independent oracle ticks.
    Returns the grid width (CTAs per robot) of the traced first tick."""
    R = x0.shape[0]
    b.engine.set_trace(True)
    x0_d = _dev(x0)
    U, idx = np.zeros((R, sp.T, 2)), np.zeros(R, dtype=int)
    width = None
    for tick in range(ticks):
        u0 = b.step(x0_d).cpu().numpy()
        Unew, inew = b.nominal(), b.waypoint_idx()
        if width is None:
            width = len(b.engine.trace()[0])
        for r in robots:
            o = _oracle_tick(b.engine, sp, path, U[r], idx[r], x0[r], b.seed, tick, robot=int(r))
            assert np.max(np.abs(Unew[r] - o["U_after"])) <= tol, (tick, r, np.max(np.abs(Unew[r] - o["U_after"])))
            assert np.max(np.abs(u0[r] - o["u0"])) <= tol, (tick, r)
            assert inew[r] == o["idx_after"], (tick, r)
        U, idx = Unew.astype(np.float64), inew
    return width


def _rc_fleet(R, K, T, obstacles, seed):
    from mppi_b200.batched import BatchedMPPI
    path = Golden("racecar_noobs").path
    sp = orc.racecar_spec(K=K, T=T, obstacles=obstacles, dtype=np.float64)
    b = BatchedMPPI(R, path, model="bicycle", delta_t=0.05, max_u=(0.523, 2.0), num_samples_K=K, num_horizons_T=T,
                    param_exploration=0.01, param_lambda=50.0, param_alpha=1.0, sigma=((0.5, 0.0), (0.0, 0.1)),
                    stage_cost_weight=(50.0, 50.0, 1.0, 20.0), terminal_cost_weight=(50.0, 50.0, 1.0, 20.0),
                    window=200, obstacle_circles=obstacles, margin=sp.margin, seed=seed)
    rng = np.random.default_rng(seed)
    x0 = np.stack([path[(5 * r) % 90] + rng.normal(0, [0.3, 0.3, 0.05, 0.5]) for r in range(R)])
    return b, sp, path, x0


def _rc_obstacles():
    p = Golden("racecar_noobs").path
    return np.array([[p[8, 0], p[8, 1] + 1.0, 0.8], [p[25, 0] - 0.5, p[25, 1], 0.6], [p[60, 0], p[60, 1] - 1.0, 0.8]])


def _dd_fleet(R, K, T, seed, obstacles=None, cost_mode="sum"):
    from mppi_b200.batched import BatchedMPPI
    path = Golden("diffdrive_pe0.05").path
    sp = _dd_spec(K, T, obstacles=obstacles, cost_mode=cost_mode)
    b = BatchedMPPI(R, path, num_samples_K=K, num_horizons_T=T, temperature=2.0, cost_mode=cost_mode,
                    obstacle_circles=obstacles, margin=sp.margin, seed=seed)
    return b, sp, path, _fleet_states(path, R, seed)


@pytest.mark.parametrize("R", [2, 3])
def test_two_level_merge_per_robot_matches_oracle(R):
    b, sp, path, x0 = _dd_fleet(R, 65536, 30, seed=31)
    width = _fleet_vs_oracle(b, sp, path, x0, range(R), U_ATOL_DD)
    # >= 64 CTAs per robot: the per-robot group tickets and group partials run (the last group of 16 is ragged unless
    # the width is a multiple of 16)
    assert width >= 64, width
    b.engine.close()


def test_batched_bicycle_footprint_obstacles_long_window_matches_oracle():
    b, sp, path, x0 = _rc_fleet(2, 32768, 50, _rc_obstacles(), seed=32)
    width = _fleet_vs_oracle(b, sp, path, x0, range(2), U_ATOL_RC)
    assert width >= 64, width
    b.engine.close()


@pytest.mark.parametrize("case", ["bicycle_footprint", "diffdrive_circle", "diffdrive_last"])
def test_one_cta_per_robot_fleets_match_oracle(case):
    R, K = 300, 1024
    if case == "bicycle_footprint":
        b, sp, path, x0 = _rc_fleet(R, K, 30, _rc_obstacles(), seed=33)
        tol = U_ATOL_RC
    else:
        p = Golden("diffdrive_pe0.05").path
        obs = np.array([[p[i, 0] + 0.3, p[i, 1], 0.4] for i in (30, 80, 130)]) if case == "diffdrive_circle" else None
        b, sp, path, x0 = _dd_fleet(R, K, 30, seed=34, obstacles=obs, cost_mode="last" if case == "diffdrive_last" else "sum")
        tol = U_ATOL_DD
    robots = np.random.default_rng(35).choice(R, 8, replace=False)
    width = _fleet_vs_oracle(b, sp, path, x0, robots, tol)
    assert width == 1, width                        # the stash kernel, no ticket, the robot's CTA finalizes alone
    b.engine.close()


# ---- D. rollout-selection boundaries ----------------------------------------------------------------------------------
FAMILIES = {"diffdrive_static": (lambda T: _dd_case(65536, T), "stash", (30, 50), U_ATOL_DD),
            "racecar_obstacles": (lambda T: _rc_case(16384, T), "tpar", (50,), U_ATOL_RC)}


@pytest.mark.parametrize("family", list(FAMILIES))
def test_rollout_path_selection_has_no_holes_and_both_sides_match_oracle(family, capfd):
    case, fast, headline, tol = FAMILIES[family]
    chosen = {}
    for T in range(10, 129):
        sp, path, x0 = case(T)
        eng, sel, grid = _create(sp, path, capfd)
        eng.set_trace(True)
        eng.step(x0, None, seed=3, tick=0)
        width = len(eng.trace()[0])
        eng.close()
        assert width == grid, (T, sel, grid, width)            # the Philox tick ran the grid of the path selected
        if sel == "tpar":
            assert -(-sp.K // width) <= 64, (T, width)          # time-parallel CTAs own <= 64 samples
        chosen[T] = sel
    with_fast = [T for T in chosen if chosen[T] == fast]
    # one contiguous range from the smallest horizon: a hole (like the lost stash at T = 18..23) is a silent slow-down
    assert with_fast == list(range(10, 10 + len(with_fast))), (family, chosen)
    assert all(T in with_fast for T in headline), (family, chosen)
    edge = 10 + len(with_fast)                                   # first horizon without the fast path
    for T in sorted({16, 17, 23, 24, edge - 1, edge, 128} & set(range(10, 129))):
        sp, path, x0 = case(T)
        h = _Handle(sp, path, x0, tol)
        h.eng.set_nominal((np.random.default_rng(T).normal(0, 0.2, (T, 2)) * np.asarray(sp.u_max) * 0.5).astype(np.float32))
        h.U = h.eng.get_nominal().astype(np.float64)
        h.step_and_check()
        h.eng.close()


def test_tpar_sample_count_boundary_matches_oracle_and_serial_kernel(capfd):
    """K = 296 * 64 is the largest sample count whose CTAs own <= 64 samples on 296 CTAs: time-parallel; one more
    sample: the serial stash kernel.  Both against the oracle and against each other on the samples they share."""
    T, n_sm = 50, torch.cuda.get_device_properties(0).multi_processor_count
    k_tpar = 2 * n_sm * 64
    res = {}
    for K, want in ((k_tpar, "tpar"), (k_tpar + 1, "stash")):
        sp, path, x0 = _rc_case(K, T)
        eng, sel, _ = _create(sp, path, capfd)
        assert sel == want, (K, sel)
        eng.set_keep_costs(True)
        u0, useq = eng.step(x0, None, seed=5, tick=2)
        useq = useq.copy()
        d_traj = torch.zeros(K, T, 4, device="cuda")
        d_cost = torch.zeros(K, device="cuda")
        d_idx = torch.zeros(K, dtype=torch.int32, device="cuda")
        eng.top_trajectories(x0, d_traj, K, d_idx=d_idx, d_cost=d_cost, seed=5, tick=2)
        S = np.empty(K, dtype=np.float32)
        S[d_idx.cpu().numpy()] = d_cost.cpu().numpy()
        o = _oracle_tick(eng, sp, path, np.zeros((T, 2)), 0, x0, 5, 2)
        assert np.max(np.abs(useq - o["U_after"])) <= U_ATOL_RC, (K, np.max(np.abs(useq - o["U_after"])))
        assert eng.get_waypoint_idx() == o["idx_after"]
        res[K] = (S, sp.n_exploit())
        eng.close()
    (Sa, na), (Sb, nb) = res[k_tpar], res[k_tpar + 1]
    # same Philox stream per sample index; a sample is exploit / explore by the global threshold, which moves with K
    same = np.ones(k_tpar, dtype=bool)
    same[min(na, nb):max(na, nb)] = False
    assert np.allclose(Sa[same], Sb[:k_tpar][same], rtol=2e-6, atol=1e-6), np.max(np.abs(Sa[same] - Sb[:k_tpar][same]))


# ---- E. the drop-in classes only the engine replayed so far ---------------------------------------------------------------
def test_race_car_class_replays_its_golden_and_raises_at_the_path_end():
    from mppi_b200.mppi_race_car import MPPIRacecarController
    g = Golden("racecar_noobs")
    m = g.meta
    rc = MPPIRacecarController(horizon_step_T=m["horizon_step_T"], number_of_samples_K=m["number_of_samples_K"],
                               param_alpha=m["param_alpha"], visualize_optimal_traj=False, visualze_sampled_trajs=False)
    rc.ref_path = g.path
    for i in range(g.n_ticks):
        u0, u, traj, samp = rc._calc_control_input(g.rec["x0"][i], noise=g.eps[i])
        assert np.max(np.abs(u - g.rec["U_after"][i])) <= U_ATOL_DD, (i, np.max(np.abs(u - g.rec["U_after"][i])))
        assert np.max(np.abs(u0 - g.rec["u0"][i])) <= U_ATOL_DD, i
        assert rc.prev_waypoints_idx == int(g.rec["idx_after"][i]), i
    # the reference raises once the nominal index reaches the last waypoint (mppi_race_car.py:65), not before
    n = g.path.shape[0]
    rc.prev_waypoints_idx = n - 6
    for j in range(n - 5, n - 1):
        rc._calc_control_input(g.path[j])
        assert rc.prev_waypoints_idx == j
    with pytest.raises(IndexError):
        rc._calc_control_input(g.path[n - 1])
    assert rc.prev_waypoints_idx == n - 1
    rc.engine.close()


def test_diff_drive_obstacle_class_replays_its_golden():
    from mppi_b200.mppi_differential_drive_obs import MPPIAlgorithms
    g = Golden("diffdrive_obs")
    m = g.meta
    ctrl = MPPIAlgorithms(
        delta_t=m["delta_t"], ref_path=g.path, max_speed=m["max_speed"], max_omega=m["max_omega"],
        num_samples_K=m["num_samples_K"], num_horizons_T=m["num_horizons_T"], param_exploration=m["param_exploration"],
        param_lambda=m["param_lambda"], param_alpha=m["param_alpha"], sigma=np.array([[0.1, 0.0], [0.0, 0.01]]),
        stage_cost_weight=10 * np.array([5.0, 6.0, 9.0]), terminal_cost_weight=10 * np.array([5.0, 6.0, 9.0]),
        obstacle_circles=g.obstacles, safety_margin_rate=m["safety_margin_rate"],
        visualize_optimal_traj=False, visualze_sampled_trajs=False)
    assert ctrl.safefy_margin_rate == m["safety_margin_rate"]
    for i in range(g.n_ticks):
        u0, u, traj, samp = ctrl._calc_input_control(g.rec["x0"][i], noise=g.eps[i])
        assert np.max(np.abs(u - g.rec["U_after"][i])) <= U_ATOL_DD, (i, np.max(np.abs(u - g.rec["U_after"][i])))
        assert np.max(np.abs(u0 - g.rec["u0"][i])) <= U_ATOL_DD, i
        assert ctrl.prev_way_point_idx == int(g.rec["idx_after"][i]), i
    ctrl.engine.close()
