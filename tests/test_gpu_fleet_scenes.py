"""Fleets in which every robot has its own goal and its own obstacle set (mppi_set_robot_goals / mppi_set_robot_obstacles,
BatchedMPPI.set_goals / set_obstacles): the scene instantiations of the tick kernel against the shared-scene kernels (bit for
bit when every robot's scene equals the shared one) and against independent C-oracle ticks fed each robot's Philox noise."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from golden_util import Golden  # noqa: E402
from oracle import c_oracle as co  # noqa: E402
from oracle import mppi_oracle as orc  # noqa: E402

U_ATOL_DD = 2e-5        # updated nominal, diff-drive (test_gpu_parity.py)
U_ATOL_RC = 1e-4        # race-car (test_gpu_config_matrix.py)
E_BADARG, E_STATE, E_UNSUPPORTED = -1, -4, -5


def _f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


def _dev(a, dtype=np.float32):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).cuda()


# ---- the supported (model, collision, cost kind) combinations, each as an oracle spec + its shared scene ------------------
def _case(kind, K, T, cost_mode="sum"):
    """(spec, path) with float32-representable shared goal / obstacles."""
    if kind in ("dd_circle_w20", "dd_circle_dyn"):
        path = Golden("diffdrive_pe0.05").path
        obs = _f32([[path[i, 0] + 0.3, path[i, 1], 0.4] for i in (30, 80, 130)])
        sp = orc.diffdrive_spec(K=K, T=T, param_exploration=0.05, cost_mode=cost_mode, waypoint_mode="frozen",
                                obstacles=obs, margin=1.2)
        sp.temperature = 2.0
        if kind == "dd_circle_dyn":
            sp.window = 64
        return sp, path
    if kind in ("rc_footprint_dyn", "rc_footprint_w20"):
        path = Golden("racecar_noobs").path
        obs = _f32([[path[8, 0], path[8, 1] + 1.0, 0.8], [path[25, 0] - 0.5, path[25, 1], 0.6], [path[60, 0], path[60, 1] - 1.0, 0.8]])
        sp = orc.racecar_spec(K=K, T=T, obstacles=obs, dtype=np.float64)
        sp.cost_mode = cost_mode
        if kind == "rc_footprint_w20":
            sp.window = 20
        return sp, path
    if kind in ("goal_none", "goal_circle"):
        sp = orc.goal_spec(K, T, [5.0, 5.0], cost_mode=cost_mode, obstacles=None if kind == "goal_circle" else np.zeros((0, 3)))
        sp.temperature = 5.0
        return sp, None
    assert kind == "target_soft"
    sp = orc.target_soft_spec(K, T, dtype=np.float64)
    sp.cost_mode = cost_mode
    sp.obstacles, sp.obs_vel = _f32(sp.obstacles), _f32(sp.obs_vel)
    return sp, None


KINDS = ["dd_circle_w20", "dd_circle_dyn", "rc_footprint_dyn", "rc_footprint_w20", "goal_none", "goal_circle", "target_soft"]


def _fleet(sp, path, R, seed):
    from mppi_b200.batched import BatchedMPPI
    goal = None if sp.cost_kind == "path" else sp.goal[:2 if sp.cost_kind == "goal" else 3]
    b = BatchedMPPI(R, path, model=sp.model, delta_t=sp.dt, max_u=sp.u_max, num_samples_K=sp.K, num_horizons_T=sp.T,
                    param_exploration=sp.param_exploration, param_lambda=sp.param_lambda, param_alpha=sp.param_alpha,
                    sigma=sp.sigma, stage_cost_weight=sp.stage_w, terminal_cost_weight=sp.term_w, temperature=sp.temperature,
                    cost_mode=sp.cost_mode, window=sp.window,
                    obstacle_circles=sp.obstacles if sp.collision != "none" else None, margin=sp.margin, seed=seed,
                    cost_kind=sp.cost_kind, goal=goal, collision=sp.collision, filter_kind=sp.filter_kind,
                    ctrl_w=sp.ctrl_w, soft_obs_weight=sp.soft_w, soft_obs_safety=sp.soft_sd)
    if sp.cost_kind == "target_soft":
        b.engine.set_moving_obstacles(sp.obstacles, sp.obs_vel)
    return b


def _states(sp, path, R, seed):
    rng = np.random.default_rng(seed)
    if sp.model == "bicycle":
        return np.stack([path[(5 * r) % 90] + rng.normal(0, [0.3, 0.3, 0.05, 0.5]) for r in range(R)])
    if path is not None:
        return np.stack([np.append(path[(7 * r) % 140, :2] + rng.normal(0, 0.1, 2), path[(7 * r) % 140, 2] + rng.normal(0, 0.1))
                         for r in range(R)])
    return np.stack([np.array([0.5, 0.3, 0.2]) + rng.normal(0, [0.5, 0.5, 0.3]) for r in range(R)])


def _shared_rows(sp, R):
    """Per-robot tables that repeat the shared scene in every slot."""
    goals = None
    if sp.cost_kind != "path":
        goals = np.tile(_f32(sp.goal[:2 if sp.cost_kind == "goal" else 3]), (R, 1))
    obs = None
    if sp.cost_kind == "target_soft":
        obs = np.tile(np.hstack([sp.obstacles, sp.obs_vel])[None], (R, 1, 1))
    elif sp.collision != "none":
        obs = np.tile(sp.obstacles[None], (R, 1, 1))
    return goals, obs


def _run(b, x0, ticks):
    out = []
    x0_d = _dev(x0)
    for _ in range(ticks):
        u0 = b.step(x0_d).clone()
        out.append((u0.cpu().numpy(), b.nominal(), b.waypoint_idx()))
    return out


def _assert_same(got, ref, where):
    for i, ((u, U, idx), (u2, U2, idx2)) in enumerate(zip(got, ref)):
        assert np.array_equal(u, u2), (where, i, np.max(np.abs(u - u2)))
        assert np.array_equal(U, U2), (where, i)
        assert np.array_equal(idx, idx2), (where, i)


# ---- 1. the same scene in every slot is the shared scene, bit for bit ------------------------------------------------------
@pytest.mark.parametrize("T", [30, 128])              # noise stash / regenerate-noise path
@pytest.mark.parametrize("R", [6, 300])               # several CTAs per robot (ticket merge) / one CTA per robot
@pytest.mark.parametrize("cost_mode", ["last", "sum"])
@pytest.mark.parametrize("kind", KINDS)
def test_same_scene_in_every_slot_is_bit_identical_to_the_shared_scene(kind, cost_mode, R, T):
    sp, path = _case(kind, 1024, T, cost_mode)
    x0 = _states(sp, path, R, 41)
    ref = _fleet(sp, path, R, 41)
    want = _run(ref, x0, 3)
    ref.engine.close()
    b = _fleet(sp, path, R, 41)
    goals, obs = _shared_rows(sp, R)
    if goals is not None:
        b.set_goals(goals)
    if obs is not None:
        b.set_obstacles(obs)
    _assert_same(_run(b, x0, 3), want, (kind, cost_mode, R, T))
    assert b.engine.check_guards() == 0
    b.engine.close()


@pytest.mark.parametrize("component", ["goals", "obstacles"])
def test_one_component_per_robot_and_the_other_shared(component):
    sp, _ = _case("goal_circle", 1024, 30)
    R = 6
    x0 = _states(sp, None, R, 42)
    ref = _fleet(sp, None, R, 42)
    want = _run(ref, x0, 3)
    ref.engine.close()
    b = _fleet(sp, None, R, 42)
    goals, obs = _shared_rows(sp, R)
    if component == "goals":
        b.set_goals(_dev(goals))
    else:
        b.set_obstacles(_dev(obs), counts=_dev(np.full(R, obs.shape[1]), np.int32))
    _assert_same(_run(b, x0, 3), want, component)
    b.engine.close()


def test_time_parallel_handle_runs_its_scene_ticks_on_the_stash_path(capfd):
    """One race-car robot (window 200, sum): its shared-scene Philox ticks are time-parallel.  Its scene ticks take the stash
    kernel with the stash grid -- the grid mppi_step_batched gives its shared-scene ticks -- so the two are bit-identical; the
    closed loop (time-parallel with the shared scene) follows the oracle with a per-robot scene."""
    import os
    import re
    sp, path = _case("rc_footprint_dyn", 16384, 30)
    x0 = _states(sp, path, 1, 51)
    ref = _fleet(sp, path, 1, 51)
    want = _run(ref, x0, 2)
    ref.engine.close()
    capfd.readouterr()
    os.environ["MPPI_VERBOSE"] = "1"
    try:
        b = _fleet(sp, path, 1, 51)
        goals, obs = _shared_rows(sp, 1)
        b.set_obstacles(obs)
    finally:
        del os.environ["MPPI_VERBOSE"]
    err = capfd.readouterr().err
    assert re.search(r"rollout path tpar", err) and re.search(r"scene ticks take the stash path", err), err
    _assert_same(_run(b, x0, 2), want, "tpar handle")
    b.engine.close()
    b = _fleet(sp, path, 1, 52)
    x2, _, obs, counts = _distinct_scene(sp, path, 2, 51)          # robot 0 of a 2-robot scene starts at x0[0]
    assert np.array_equal(x2[0], x0[0])
    obs, counts = obs[:1], counts[1:2]                               # 16 obstacles around it
    b.set_obstacles(obs, counts=counts)
    n = 4
    states, _ = b.run_closed_loop(x0, n)
    s_r = _robot_spec(sp, None, obs, counts, 0)
    xs, _, _, _ = _oracle_loop(b, s_r, path, x0[0], 0, n, lambda x, u: orc.plant_bicycle(x, u, sp.dt))
    assert np.max(np.abs(states - xs)) <= 5e-4, np.max(np.abs(states - xs))
    b.engine.close()


# ---- 2. distinct scenes against the oracle -----------------------------------------------------------------------------------
def _distinct_scene(sp, path, R, seed):
    """Per-robot goals, obstacle rows (R, 16, ncol) and counts (0 and 16 included), float32-representable."""
    rng = np.random.default_rng(seed)
    x0 = _states(sp, path, R, seed)
    goals = None
    if sp.cost_kind == "goal":
        goals = _f32(x0[:, :2] + rng.uniform(2.0, 5.0, (R, 2)))
    elif sp.cost_kind == "target_soft":
        goals = _f32(np.hstack([x0[:, :2] + rng.uniform(2.0, 5.0, (R, 2)), rng.uniform(0.0, 3.0, (R, 1))]))
    if sp.cost_kind == "target_soft":
        obs = np.concatenate([x0[:, None, :2] + rng.uniform(-3.0, 5.0, (R, 16, 2)), rng.normal(0, 0.3, (R, 16, 2))], axis=2)
    else:
        obs = np.concatenate([x0[:, None, :2] + rng.uniform(-4.0, 6.0, (R, 16, 2)), rng.uniform(0.2, 0.9, (R, 16, 1))], axis=2)
    counts = rng.integers(1, 16, R).astype(np.int32)
    counts[0], counts[1] = 0, 16
    return x0, goals, _f32(obs), counts


def _robot_spec(sp, goals, obs, counts, r):
    import copy
    s = copy.deepcopy(sp)
    if goals is not None:
        s.goal = np.zeros(3)
        s.goal[:goals.shape[1]] = goals[r]
    rows = obs[r, :counts[r]]
    if sp.cost_kind == "target_soft":
        s.obstacles, s.obs_vel = rows[:, :2].copy(), rows[:, 2:].copy()
    else:
        s.obstacles = rows.copy()
        if s.collision == "none" and rows.shape[0]:
            s.collision = "circle"
    return s


DISTINCT = {"goal_circle": (lambda: _case("goal_circle", 1024, 30), U_ATOL_DD),
            "rc_footprint_dyn": (lambda: _case("rc_footprint_dyn", 1024, 30), U_ATOL_RC),
            "target_soft": (lambda: _case("target_soft", 1024, 30), U_ATOL_DD)}


@pytest.mark.parametrize("name", list(DISTINCT))
def test_distinct_scenes_match_independent_oracle_ticks(name):
    make, tol = DISTINCT[name]
    sp, path = make()
    R = 6
    x0, goals, obs, counts = _distinct_scene(sp, path, R, 43)
    b = _fleet(sp, path, R, 43)
    if goals is not None:
        b.set_goals(goals)
    b.set_obstacles(obs, counts=counts)
    specs = [_robot_spec(sp, goals, obs, counts, r) for r in range(R)]
    x0_d = _dev(x0)
    eps = torch.zeros(sp.K, sp.T, 2, dtype=torch.float32, device="cuda")
    U, idx = np.zeros((R, sp.T, 2)), np.zeros(R, dtype=int)
    first = None
    for tick in range(2):
        u0 = b.step(x0_d).cpu().numpy()
        first = u0 if first is None else first
        Unew, inew = b.nominal(), b.waypoint_idx()
        for r in range(R):
            b.engine.generate_noise(eps, seed=43, tick=tick, robot=r)
            o = co.tick(specs[r], path, U[r], int(idx[r]), _f32(x0[r]), eps.cpu().numpy())
            assert np.max(np.abs(Unew[r] - o["U_after"])) <= tol, (name, tick, r, np.max(np.abs(Unew[r] - o["U_after"])))
            assert np.max(np.abs(u0[r] - o["u0"])) <= tol, (name, tick, r)
            if path is not None:
                assert inew[r] == o["idx_after"], (name, tick, r)
        U, idx = Unew.astype(np.float64), inew
    assert b.engine.check_guards() == 0
    b.engine.close()
    # the scenes matter: the same fleet with the shared scene steers differently
    shared = _fleet(sp, path, R, 43)
    u_shared = shared.step(x0_d).cpu().numpy()
    shared.engine.close()
    assert not np.array_equal(u_shared, first), name


# ---- 3. closed loop, then new goals / obstacles on the same handle ----------------------------------------------------------
def _oracle_loop(b, sp, path, x0, r, n, plant, tick_base=0, U=None, idx=0):
    eps = torch.zeros(sp.K, sp.T, 2, dtype=torch.float32, device="cuda")
    x = _f32(x0)
    U = np.zeros((sp.T, 2)) if U is None else U
    xs, us = [x.copy()], []
    for i in range(n):
        b.engine.generate_noise(eps, seed=b.seed, tick=tick_base + i, robot=r)
        o = co.tick(sp, path, U, idx, _f32(x), eps.cpu().numpy())
        U, idx = o["U_after"], o["idx_after"]
        x = plant(x, o["u0"])
        xs.append(x.copy()); us.append(o["u0"].copy())
    return np.array(xs), np.array(us), U, idx


@pytest.mark.parametrize("name", ["goal_circle", "rc_footprint_dyn"])
def test_closed_loop_with_distinct_scenes_follows_reinstalled_scenes(name):
    sp, path = _case(name, 1024, 20)
    R, n = 6, 12
    x0, goals, obs, counts = _distinct_scene(sp, path, R, 44)
    b = _fleet(sp, path, R, 44)
    if goals is not None:
        b.set_goals(goals)
    b.set_obstacles(obs, counts=counts)
    plant = (lambda x, u: orc.plant_bicycle(x, u, sp.dt)) if sp.model == "bicycle" else (lambda x, u: orc.plant_diffdrive(x, u, sp.dt))
    states, controls = b.run_closed_loop(x0, n)
    ends = []
    for r in range(R):
        s_r = _robot_spec(sp, goals, obs, counts, r)
        xs, us, U, idx = _oracle_loop(b, s_r, path, x0[r], r, n, plant)
        assert np.max(np.abs(states[:, r] - xs)) <= 5e-4, (name, r, np.max(np.abs(states[:, r] - xs)))
        assert np.max(np.abs(controls[:, r] - us)) <= 2e-4, (name, r)
        ends.append((U, idx))
    # a different scene for the second call on the same handle (same graph: the table's address does not change)
    rng = np.random.default_rng(45)
    if goals is not None:
        goals2 = _f32(goals + rng.uniform(-2.0, 2.0, goals.shape))
        b.set_goals(goals2)
        obs2, counts2 = obs, counts
    else:
        goals2 = None
        obs2 = _f32(np.concatenate([obs[..., :2] + rng.uniform(-1.0, 1.0, obs[..., :2].shape), obs[..., 2:]], axis=2))
        counts2 = counts[::-1].copy()
        b.set_obstacles(obs2, counts=counts2)
    states2, _ = b.run_closed_loop(states[-1], n)
    for r in range(R):
        s_r = _robot_spec(sp, goals2, obs2, counts2, r)
        xs2, _, _, _ = _oracle_loop(b, s_r, path, states[-1, r].astype(np.float64), r, n, plant, tick_base=n,
                                    U=ends[r][0], idx=ends[r][1])
        assert np.max(np.abs(states2[:, r] - xs2)) <= 2e-3, (name, r, np.max(np.abs(states2[:, r] - xs2)))
    assert b.engine.check_guards() == 0
    b.engine.close()


# ---- 4. stream order: goals written by torch on the device every tick, no synchronisation -----------------------------------
def test_goals_written_on_the_device_every_tick_are_consumed_in_stream_order():
    sp, _ = _case("goal_circle", 4096, 30)
    R = 64
    x0 = _dev(_states(sp, None, R, 46))
    base = _dev(np.random.default_rng(46).uniform(2.0, 6.0, (R, 2)))

    def run(sync):
        b = _fleet(sp, None, R, 46)
        g = torch.empty_like(base)
        out = []
        for i in range(5):
            torch.mul(base, 1.0 + 0.1 * i, out=g)            # overwrite the buffer the previous install read
            if sync:
                torch.cuda.synchronize()
            b.set_goals(g)
            if sync:
                torch.cuda.synchronize()
            out.append(b.step(x0).clone())
            if sync:
                torch.cuda.synchronize()
        res = torch.stack(out).cpu().numpy()
        b.engine.close()
        return res

    fast, slow = run(False), run(True)
    assert np.array_equal(fast, slow)
    assert np.all(np.isfinite(fast)) and np.max(np.abs(fast[0] - fast[4])) > 0.0


# ---- 5. back to the shared scene, and every refusal -------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["goal_circle", "target_soft"])
def test_use_shared_scene_restores_the_shared_fleet(kind):
    """Back to the shared goal and obstacles, including a target_soft fleet's shared moving obstacles set on its engine."""
    sp, _ = _case(kind, 1024, 30)
    R = 6
    x0 = _states(sp, None, R, 47)
    ref = _fleet(sp, None, R, 47)
    want = _run(ref, x0, 2)
    ref.engine.close()
    b = _fleet(sp, None, R, 47)
    _, goals, obs, counts = _distinct_scene(sp, None, R, 47)
    b.set_goals(goals)
    b.set_obstacles(obs, counts=counts)
    b.use_shared_scene()
    _assert_same(_run(b, x0, 2), want, "shared again")
    assert b.engine.check_guards() == 0
    b.engine.close()


def test_refusals():
    from mppi_b200 import _lib
    from mppi_b200.engine import MPPIEngine
    from gpu_util import engine_from_spec
    lib = _lib.load()
    obs3 = _dev(np.zeros((2, 4, 3)))
    obs4 = _dev(np.zeros((2, 4, 4)))
    g2, g3 = _dev(np.zeros((2, 2))), _dev(np.zeros((2, 3)))
    p = C.c_void_p

    def robot_obs(eng, t, m, ncol):
        return lib.mppi_set_robot_obstacles(eng._h, p(t.data_ptr()), None, m, ncol)

    def robot_goals(eng, t, n):
        return lib.mppi_set_robot_goals(eng._h, p(t.data_ptr()), n)

    # path fleet with circles: no goal; bad shapes
    sp, path = _case("dd_circle_w20", 256, 30)
    eng = engine_from_spec(sp, path, n_robots=2)
    assert robot_goals(eng, g2, 2) == E_STATE
    assert robot_obs(eng, obs4, 4, 4) == E_STATE                 # moving obstacles belong to target_soft
    assert robot_obs(eng, obs3, 17, 3) == E_BADARG and robot_obs(eng, obs3, -1, 3) == E_BADARG
    assert robot_obs(eng, obs3, 4, 5) == E_BADARG
    assert lib.mppi_set_robot_obstacles(eng._h, None, None, 4, 3) == E_BADARG
    assert robot_obs(eng, obs3, 4, 3) == 0
    assert eng.check_guards() == 0
    eng.close()
    # goal fleet without obstacles: no circles; goal width
    sp, _ = _case("goal_none", 256, 30)
    eng = engine_from_spec(sp, None, n_robots=2)
    assert robot_obs(eng, obs3, 4, 3) == E_STATE and robot_obs(eng, obs4, 4, 4) == E_STATE
    assert robot_goals(eng, g3, 3) == E_BADARG and robot_goals(eng, g2, 4) == E_BADARG
    assert lib.mppi_set_robot_goals(eng._h, None, 2) == E_BADARG
    eng.close()
    # target_soft: no static circles
    sp, _ = _case("target_soft", 256, 30)
    eng = engine_from_spec(sp, None, n_robots=2)
    assert robot_obs(eng, obs3, 4, 3) == E_STATE and robot_goals(eng, g2, 2) == E_BADARG
    assert robot_obs(eng, obs4, 4, 4) == 0 and robot_goals(eng, g3, 3) == 0
    eng.close()
    # strict waypoint mode, learned dynamics, a combination without a scene kernel
    sp, path = _case("dd_circle_w20", 256, 30)
    sp.waypoint_mode = "strict"
    eng = engine_from_spec(sp, path)
    assert robot_obs(eng, _dev(np.zeros((1, 4, 3))), 4, 3) == E_UNSUPPORTED
    eng.close()
    mlp = MPPIEngine(model="diffdrive_mlp", K=256, T=30, dt=0.1, u_max=(5.0, 3.14), sigma=np.diag([0.1, 0.01]),
                     stage_w=(5, 5, 10), term_w=(5, 5, 10), param_exploration=0.05, param_lambda=1.0, param_alpha=0.2,
                     temperature=2.0, window=20, cost_mode="sum", waypoint_mode="frozen", filter_kind="diffdrive", yaw_wrap=False)
    assert robot_goals(mlp, _dev(np.zeros((1, 2))), 2) == E_UNSUPPORTED
    mlp.close()
    sp, path = _case("rc_footprint_dyn", 256, 30)
    sp.collision = "circle"
    eng = engine_from_spec(sp, path, n_robots=2)
    assert robot_obs(eng, obs3, 4, 3) == E_UNSUPPORTED              # bicycle + circles: no scene instantiation
    eng.close()
    # one robot with a per-robot goal installed: every tick entry point but the fleet ones refuses
    sp, _ = _case("goal_circle", 256, 30)
    eng = engine_from_spec(sp, None)
    eng.set_keep_costs(True)
    assert robot_goals(eng, _dev(np.array([[4.0, 4.0]])), 2) == 0
    x0 = (C.c_double * 4)(0.0, 0.0, 0.0, 0.0)
    S = torch.zeros(256, device="cuda")
    assert lib.mppi_step(eng._h, x0, None, 0, 0, None, None) == E_STATE
    assert b"per-robot" in lib.mppi_last_error(eng._h)
    assert lib.mppi_step_async(eng._h, x0, None, 0, 0) == E_STATE
    assert lib.mppi_rollout_costs(eng._h, x0, None, 0, 0, p(S.data_ptr())) == E_STATE
    assert lib.mppi_reduce_update(eng._h, p(S.data_ptr()), None, 0, 0, None, None, None) == E_STATE
    assert lib.mppi_get_trajectories(eng._h, x0, None, 0, 0, None, None) == E_STATE
    traj = torch.zeros(4, 30, 3, device="cuda")
    assert lib.mppi_get_top_trajectories(eng._h, x0, None, 0, 0, 4, 1, None, p(traj.data_ptr()), None, None) == E_STATE
    uid = C.create_string_buffer(128)
    assert lib.mppi_comm_init(eng._h, uid, 0, 1) == E_STATE
    assert lib.mppi_comm_p2p_export(eng._h, 2, C.create_string_buffer(64)) == E_STATE
    # the fleet entry points run it; the shared setter lifts the refusal
    states, _ = eng.run_closed_loop(np.zeros(3), 3)
    assert np.all(np.isfinite(states))
    eng.set_goal([4.0, 4.0])
    eng.step(np.zeros(3), None, 0, 0)
    assert eng.check_guards() == 0
    eng.close()


# ---- 6. scale: 4096 robots with their own circle sets ------------------------------------------------------------------------
def _big_fleet(seed):
    sp, path = _case("dd_circle_w20", 1024, 30)
    R = 4096
    b = _fleet(sp, path, R, seed)
    rng = np.random.default_rng(seed)
    x0 = np.stack([np.append(path[r % 100, :2] + rng.normal(0, 0.1, 2), path[r % 100, 2] + rng.normal(0, 0.1)) for r in range(R)])
    b.engine.set_waypoint_idx(np.arange(R) % 100)
    around = np.array([path[(r % 100 + 5) % 168, :2] for r in range(R)])
    obs = _f32(np.concatenate([around[:, None, :] + rng.uniform(-3.0, 3.0, (R, 16, 2)), rng.uniform(0.2, 0.6, (R, 16, 1))], axis=2))
    counts = rng.integers(4, 17, R).astype(np.int32)
    b.set_obstacles(obs, counts=counts)
    return b, sp, path, x0, obs, counts


def test_4096_robot_fleet_with_own_obstacle_sets_one_launch_per_tick_subset_vs_oracle():
    b, sp, path, x0, obs, counts = _big_fleet(48)
    R = x0.shape[0]
    x0_d = _dev(x0)
    l0 = b.engine.timings()["launches"]
    u0 = b.step(x0_d).cpu().numpy()
    b.engine.synchronize()
    assert b.engine.timings()["launches"] - l0 == 1
    Unew, inew = b.nominal(), b.waypoint_idx()
    eps = torch.zeros(sp.K, sp.T, 2, dtype=torch.float32, device="cuda")
    for r in np.random.default_rng(48).choice(R, 4, replace=False):
        s_r = _robot_spec(sp, None, obs, counts, r)
        b.engine.generate_noise(eps, seed=48, tick=0, robot=int(r))
        o = co.tick(s_r, path, np.zeros((sp.T, 2)), int(r % 100), _f32(x0[r]), eps.cpu().numpy())
        assert np.max(np.abs(Unew[r] - o["U_after"])) <= U_ATOL_DD, (r, np.max(np.abs(Unew[r] - o["U_after"])))
        assert np.max(np.abs(u0[r] - o["u0"])) <= U_ATOL_DD and inew[r] == o["idx_after"]
    b.engine.close()
    b, sp, path, x0, obs, counts = _big_fleet(49)
    n = 10
    l0 = b.engine.timings()["launches"]
    states, controls = b.run_closed_loop(x0, n)
    assert b.engine.timings()["launches"] - l0 == n                     # one launch per tick for the whole fleet
    assert np.all(np.isfinite(states)) and np.all(np.isfinite(controls))
    plant = lambda x, u: orc.plant_diffdrive(x, u, sp.dt)              # noqa: E731
    for r in np.random.default_rng(49).choice(R, 3, replace=False):
        s_r = _robot_spec(sp, None, obs, counts, r)
        xs, us, _, _ = _oracle_loop(b, s_r, path, x0[r], int(r), 6, plant, idx=int(r % 100))
        assert np.max(np.abs(states[:7, r] - xs)) <= 1e-3, (r, np.max(np.abs(states[:7, r] - xs)))
        assert np.max(np.abs(controls[:6, r] - us)) <= 5e-4, r
    assert b.engine.check_guards() == 0
    b.engine.close()


_FP32_NOMINAL_TFLOPS = 71.0          # what the FFMA probe measures on an unthrottled B200 (test_gpu_perf_guard.py)


def _clock_scale():
    import mppi_b200
    v = C.c_double(0.0)
    rc = mppi_b200.load().mppi_probe_fp32_peak(0, 0, C.byref(v))
    assert rc == 0 and v.value > 0.0, (rc, v.value)
    return max(1.0, _FP32_NOMINAL_TFLOPS / v.value)


def test_4096_robot_scene_fleet_tick_stays_under_its_device_time_bound():
    """4096 robots x K = 1024 x T = 30, every robot with its own 4-16 circles: BOUND_MS per tick (about 1.7x the device time
    a B200 measures, profiles/scripts/fleet_scene.py)."""
    BOUND_MS = 2.0
    b, sp, path, x0, obs, counts = _big_fleet(50)
    x0_d = _dev(x0)
    for _ in range(5):
        b.step(x0_d)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 20
    e0.record()
    for _ in range(n):
        b.step(x0_d)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    b.engine.close()
    scale = _clock_scale()
    assert ms < BOUND_MS * scale, (ms, scale)
