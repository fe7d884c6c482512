"""Trajectory viewers of learned-dynamics controllers.  mppi_get_trajectories / mppi_get_top_trajectories replay the
tick's clamped controls (and the updated nominal) through the tick's own tcgen05 MLP rollout (the TRAJ instantiations of
mppi_mlp_rollout_kernel), so the replayed states are compared with the oracle's replay of the same controls twice, as
test_gpu_mlp.py compares costs: loosely against FP64, tightly against the device-faithful restatement with the hardware
tanh.  Row subsets keep the FP64 oracle affordable at K = 50 000; they take rows from every 128-row tile."""
import warnings
from dataclasses import replace

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from golden_util import Golden  # noqa: E402
from gpu_util import engine_from_spec  # noqa: E402
from oracle import mppi_oracle as orc  # noqa: E402
from test_gpu_mlp import hw_tanh  # noqa: E402

# Per row, the largest |state error| (m, rad) over its T = 12 steps; 99th percentile and worst row.  Measured on a B200
# (1000 W) over the 12 configurations of test_mlp_replays_match_oracle_replays: FP64 p99 <= 7.0e-5, max 1.02e-4; device-
# faithful + hardware tanh p99 <= 1.14e-5, max 1.75e-5; optimal row 1.16e-5.  The bounds leave a factor of ~3-5.
STATE_FP64_P99, STATE_FP64_MAX = 3e-4, 5e-4
STATE_HW_P99, STATE_HW_MAX = 5e-5, 8e-5
STATE_OPT = 5e-5
MPPI_E_BADARG, MPPI_E_STATE, MPPI_E_UNSUPPORTED = -1, -4, -5
X0 = np.array([0.4, 0.3, 0.5])


def _fptr(t):
    import ctypes
    return ctypes.cast(t.data_ptr(), ctypes.POINTER(ctypes.c_float))


def _mlp(n_in, n_hidden, seed=0):
    """Residual large enough to move the state by ~0.1 m per step (test_gpu_mlp._big_mlp): an error in the replayed
    model shows up far above the tight bound."""
    if n_in == 3:
        return orc.make_mlp(seed=seed, out_scale=0.5 if n_hidden == 2 else 1.5, n_in=3, n_hidden=n_hidden)
    m = orc.make_mlp(seed=seed, out_scale=0.5, n_in=5, scalers=True, scaler_gain=0.5 if n_hidden == 2 else 1.0, n_hidden=n_hidden)
    m["W0"][:, 3:] *= 8.0
    return m


def _spec(K, T, mlp):
    sp = orc.diffdrive_spec(K=K, T=T, param_exploration=0.05, cost_mode="sum", waypoint_mode="frozen", model="diffdrive_mlp",
                            mlp=mlp)
    sp.temperature = 2.0
    return sp


def _engine(sp, path):
    eng = engine_from_spec(sp, path)
    mlp = sp.mlp
    n = len([k for k in mlp if k[0] == "W" and k[1:].isdigit()])
    sc = [mlp[k] for k in ("in_mean", "in_scale", "out_mean", "out_scale")] if "in_scale" in mlp else []
    eng.set_mlp([mlp["W%d" % i] for i in range(n)], [mlp["b%d" % i] for i in range(n)], *sc)
    return eng


def _controls(sp, U, eps):
    """The clamped controls of every sample, (K, T, 2), in the device's FP32 arithmetic."""
    V = eps.astype(np.float32).copy()
    n = sp.n_exploit()
    V[:n] = (V[:n] + U[None].astype(np.float32)).astype(np.float32)
    lim = np.asarray(sp.u_max, np.float32)
    return np.clip(V, -lim, lim)


def _replay(sp, V, mode):
    """Oracle replay of exactly the controls V (n, T, 2) from X0: FP64 / device-faithful / device-faithful + hw tanh."""
    s = replace(sp, K=V.shape[0], param_exploration=1.0)          # no exploit rows: the controls are applied as given
    if mode != "fp64":
        s.mlp_precision = "f16"
        s.mlp_tanh = hw_tanh if mode == "hw" else None
    _, X = orc.rollout_states(s, np.zeros((sp.T, 2)), X0, V.astype(np.float64))
    return X


def _row_err(Xg, Xo):
    return np.abs(np.asarray(Xg, np.float64) - Xo).reshape(Xo.shape[0], -1).max(axis=1)


def _rows(K):
    if K <= 4096:
        return np.arange(K)
    return np.unique(np.concatenate([np.arange(0, K, 31), np.arange(K - 128, K)]))


def _tick(eng, sp, U, src, eps_p, eps_i):
    eng.set_nominal(U)
    eng.set_waypoint_idx(0)
    eng.step(X0, eps_i if src == "injected" else None, seed=3, tick=1)
    d_eps = eps_i if src == "injected" else None
    return d_eps, (eps_i if src == "injected" else eps_p).cpu().numpy()


def _all_sorted(eng, sp, d_eps, shift):
    K, T = sp.K, sp.T
    X = torch.zeros(K, T, 3, dtype=torch.float32, device="cuda")
    idx = torch.zeros(K, dtype=torch.int32, device="cuda")
    cost = torch.zeros(K, dtype=torch.float32, device="cuda")
    opt = eng.top_trajectories(X0, X, K, idx, cost, want_optimal=True, index_shift=shift, d_eps=d_eps, seed=3, tick=1)
    return X.cpu().numpy(), idx.cpu().numpy(), cost.cpu().numpy(), opt


def _check(report, name, err, p99, mx):
    report[name] = (float(np.quantile(err, 0.99)), float(err.max()))
    assert np.quantile(err, 0.99) <= p99 and err.max() <= mx, (name, report)


def _setup(n_in, n_hidden, K, T):
    g = Golden("diffdrive_pe0.05")
    sp = _spec(K, T, _mlp(n_in, n_hidden))
    eng = _engine(sp, g.path)
    eng.set_keep_costs(True)
    eps_p = torch.zeros(K, T, 2, dtype=torch.float32, device="cuda")
    eng.generate_noise(eps_p, seed=3, tick=1)
    eps_i = torch.zeros(K, T, 2, dtype=torch.float32, device="cuda")
    eng.generate_noise(eps_i, seed=8, tick=5)
    U = np.random.default_rng(2).normal(0, 0.5, (T, 2)).astype(np.float32)
    return g, sp, eng, eps_p, eps_i, U


@pytest.mark.parametrize("K", [300, 2048, 50000])
@pytest.mark.parametrize("n_in,n_hidden", [(3, 2), (5, 2), (3, 3), (5, 3)])
def test_mlp_replays_match_oracle_replays(n_in, n_hidden, K):
    """K = 300: a ragged tile; 2048: several tiles; 50 000: the ping-pong / two-GEMM schedules with the horizon of some
    tiles split between clusters.  Sampled rows with index_shift 1 (mppi_get_trajectories) and 0 (top-N over all K), and
    the optimal row (the clamped updated nominal), for Philox and injected noise."""
    T = 12
    g, sp, eng, eps_p, eps_i, U = _setup(n_in, n_hidden, K, T)
    rows = _rows(K)
    report = {}
    for src in ("philox", "injected"):
        d_eps, eps = _tick(eng, sp, U, src, eps_p, eps_i)
        V = _controls(sp, U, eps)
        X1 = torch.zeros(K, T, 3, dtype=torch.float32, device="cuda")
        opt1 = eng.trajectories(X0, X1, True, d_eps, seed=3, tick=1)
        X0s, idx, cost, opt0 = _all_sorted(eng, sp, d_eps, 0)
        X0u = np.empty_like(X0s)
        X0u[idx] = X0s                                           # back to sample order
        S = np.empty(K)
        S[idx] = cost
        U_pre = orc.update_vec(sp, U.astype(np.float64), S, eps.astype(np.float64), 0)["U_pre_shift"]
        lim = np.asarray(sp.u_max)
        U_pre = np.clip(U_pre, -lim, lim)
        for shift, Xg, opt in ((1, X1.cpu().numpy(), opt1), (0, X0u, opt0)):
            Vs = np.roll(V, 1, axis=1) if shift else V
            Us = np.roll(U_pre, 1, axis=0) if shift else U_pre
            for mode, p99, mx in (("fp64", STATE_FP64_P99, STATE_FP64_MAX), ("hw", STATE_HW_P99, STATE_HW_MAX)):
                _check(report, "%s shift%d %s" % (src, shift, mode), _row_err(Xg[rows], _replay(sp, Vs[rows], mode)), p99, mx)
            # the nominal is the oracle's update of the device's costs
            _check(report, "%s shift%d optimal" % (src, shift), _row_err(opt[None], _replay(sp, Us[None], "hw")),
                   STATE_OPT, STATE_OPT)
    print("replay state error n_in=%d n_hidden=%d K=%d (p99, max):" % (n_in, n_hidden, K), report)
    assert eng.check_guards() == 0
    eng.close()


@pytest.mark.parametrize("K", [2048, 50000])
@pytest.mark.parametrize("n_in,n_hidden", [(3, 2), (5, 2), (3, 3), (5, 3)])
def test_replayed_states_are_the_states_the_tick_scored(n_in, n_hidden, K):
    """With index_shift 0 a replayed row applies the controls the tick applied: FP64 costs of the replayed states and
    controls reproduce the tick's kept costs."""
    T = 12
    g, sp, eng, eps_p, eps_i, U = _setup(n_in, n_hidden, K, T)
    d_eps, eps = _tick(eng, sp, U, "philox", eps_p, eps_i)
    X, idx, cost, _ = _all_sorted(eng, sp, d_eps, 0)
    V = _controls(sp, U, eps)[idx].astype(np.float64)
    path = np.asarray(g.path, np.float64)
    Z = np.concatenate([X, X[:, -1:]], axis=1).astype(np.float64)
    s0 = eng.get_waypoint_idx()
    ref = orc._argmin_window(path, np.array(s0), sp.window, Z[..., 0], Z[..., 1])
    q = U.astype(np.float64) @ np.linalg.inv(sp.sigma)
    ctrl = sp.gamma * np.einsum("tu,ktu->kt", q, V)
    S = (orc._state_cost_vec(sp, path, Z[:, :T], ref[:, :T], sp.stage_w) + ctrl).sum(axis=1) + \
        orc._state_cost_vec(sp, path, Z[:, T], ref[:, T], sp.term_w)
    rel = np.abs(cost - S) / np.maximum(np.abs(S), 1e-9)
    print("kept cost vs replayed-state cost n_in=%d n_hidden=%d K=%d: p99 %.3g max %.3g" % (n_in, n_hidden, K, np.quantile(rel, 0.99),
                                                                                          rel.max()))
    assert np.quantile(rel, 0.99) <= 1e-5 and rel.max() <= 2e-2, (np.quantile(rel, 0.99), rel.max())
    eng.close()


@pytest.mark.parametrize("n_in,n_hidden", [(3, 2), (5, 2), (3, 3)])
def test_top_n_replays_in_cost_order(n_in, n_hidden):
    K, T = 4096, 12
    g, sp, eng, eps_p, eps_i, U = _setup(n_in, n_hidden, K, T)
    _tick(eng, sp, U, "philox", eps_p, eps_i)
    Xall = torch.zeros(K, T, 3, dtype=torch.float32, device="cuda")
    eng.trajectories(X0, Xall, False, None, seed=3, tick=1)
    Xall = Xall.cpu().numpy()
    _, idx_all, cost_all, _ = _all_sorted(eng, sp, None, 1)
    S = np.empty(K)
    S[idx_all] = cost_all
    for n_top in (1, 7, 128, 129, K // 10):
        traj = torch.zeros(n_top, T, 3, dtype=torch.float32, device="cuda")
        idx = torch.zeros(n_top, dtype=torch.int32, device="cuda")
        cost = torch.zeros(n_top, dtype=torch.float32, device="cuda")
        eng.top_trajectories(X0, traj, n_top, idx, cost, want_optimal=False, index_shift=1, seed=3, tick=1)
        got, c = idx.cpu().numpy(), cost.cpu().numpy()
        order = np.argsort(S, kind="stable")[:n_top]
        assert np.all(np.diff(c) >= 0)
        assert np.all(np.abs(S[got] - S[order]) <= 2e-5 * np.abs(S[order]) + 1e-6), (n_top, got, order)
        assert np.array_equal(c, S[got].astype(np.float32))
        # the same rows as the all-K replay, run by another schedule of the same kernel
        err = _row_err(traj.cpu().numpy(), Xall[got].astype(np.float64))
        assert err.max() <= 2 * STATE_HW_MAX, (n_top, err.max())
    eng.close()


@pytest.mark.parametrize("n_in,n_hidden", [(3, 2), (5, 2), (3, 3)])
def test_static_walk_replay_after_a_smaller_call(n_in, n_hidden, monkeypatch):
    """K = 50 000 with the whole-tile walk (MPPI_MLP_BALANCED=0, read by the library at every launch): the static ping-pong
    schedule for one GEMM per step, the static one-tile schedule for two.  A top-N call first, so the all-K call that follows
    has to grow the replay's scratch.  The static walk replays the same states as the balanced one, bit for bit."""
    K, T = 50000, 12
    g, sp, eng, eps_p, eps_i, U = _setup(n_in, n_hidden, K, T)
    _tick(eng, sp, U, "philox", eps_p, eps_i)
    X = {}
    for bal in ("0", "1"):
        monkeypatch.setenv("MPPI_MLP_BALANCED", bal)
        top = torch.zeros(K // 10, T, 3, dtype=torch.float32, device="cuda")
        idx = torch.zeros(K // 10, dtype=torch.int32, device="cuda")
        eng.top_trajectories(X0, top, K // 10, idx, want_optimal=False, index_shift=1, seed=3, tick=1)
        allk = torch.zeros(K, T, 3, dtype=torch.float32, device="cuda")
        opt = eng.trajectories(X0, allk, True, None, seed=3, tick=1)
        X[bal] = (top.cpu().numpy(), idx.cpu().numpy(), allk.cpu().numpy(), opt)
    top, idx, allk, opt = X["0"]
    rows = _rows(K)
    V = np.roll(_controls(sp, U, eps_p.cpu().numpy()), 1, axis=1)
    err = _row_err(allk[rows], _replay(sp, V[rows], "hw"))
    assert np.quantile(err, 0.99) <= STATE_HW_P99 and err.max() <= STATE_HW_MAX, (np.quantile(err, 0.99), err.max())
    assert _row_err(top, allk[idx].astype(np.float64)).max() <= 2 * STATE_HW_MAX
    for a, b in zip(X["0"], X["1"]):
        assert np.array_equal(a, b)
    assert eng.check_guards() == 0
    eng.close()


def test_device_faithful_replay_gate_catches_a_ten_percent_bias_error():
    K, T = 2048, 12
    g, sp, eng, eps_p, eps_i, U = _setup(3, 2, K, T)
    _tick(eng, sp, U, "philox", eps_p, eps_i)
    X = torch.zeros(K, T, 3, dtype=torch.float32, device="cuda")
    eng.trajectories(X0, X, False, None, seed=3, tick=1)
    V = np.roll(_controls(sp, U, eps_p.cpu().numpy()), 1, axis=1)
    wrong = {k: np.array(v, copy=True) for k, v in sp.mlp.items() if not k.startswith("_")}
    wrong["b2"] = wrong["b2"] * 1.1
    err = _row_err(X.cpu().numpy(), _replay(replace(sp, mlp=wrong), V, "hw"))
    print("replay error against a restatement with a 10 %% bias error: median %.3g" % np.quantile(err, 0.5))
    assert np.quantile(err, 0.5) > 10 * STATE_HW_P99, np.quantile(err, 0.5)
    eng.close()


def test_drop_in_class_returns_the_reference_visualisation_outputs():
    """The reference's default flags (both viewers on): optimal_traj (T,3) and sampled_traj_list (K,T,3) are the
    oracle's A16 outputs (_finish with x0 and the clamped controls, Q9 clamp of the nominal included), with no warning;
    set_sampled_top_n then returns (n_top,T,3)."""
    from mppi_b200.mppi_differential_drive import MPPIAlgorithms
    g = Golden("diffdrive_pe0.05")
    K, T = 256, 12
    mlp = _mlp(5, 2, seed=4)
    ctrl = MPPIAlgorithms(delta_t=0.1, ref_path=g.path, max_speed=5.0, max_omega=3.14, num_samples_K=K, num_horizons_T=T,
                          param_exploration=0.05, param_lambda=1.0, param_alpha=0.2, sigma=np.array([[0.1, 0.0], [0.0, 0.01]]),
                          stage_cost_weight=np.array([5.0, 5.0, 10.0]), terminal_cost_weight=np.array([5.0, 5.0, 10.0]),
                          cost_mode="sum", waypoint_mode="frozen", temperature=2.0, dynamics=mlp, seed=4)
    sp = _spec(K, T, mlp)
    sp.viz_sampled = True
    eps = torch.zeros(K, T, 2, dtype=torch.float32, device="cuda")
    ctrl.engine.generate_noise(eps, seed=4, tick=0)
    e64 = eps.cpu().numpy().astype(np.float64)
    U = np.zeros((T, 2))
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        u0, u, opt, samp = ctrl._calc_input_control(X0)
    assert opt.shape == (T, 3) and samp.shape == (K, T, 3)
    assert np.count_nonzero(opt) > 0 and np.count_nonzero(samp) > 0.9 * samp.size
    S, _, s_end = orc.costs_vec(sp, g.path, U, 0, X0, e64)
    V, _ = orc.rollout_states(sp, U, X0, e64)
    o = orc._finish(sp, U, S, e64, s_end, x0=X0, V=V)
    e_opt = _row_err(opt[None], o["optimal_traj"][None])
    e_samp = _row_err(samp, o["sampled_traj"])
    print("drop-in replay error: optimal %.3g, sampled p99 %.3g max %.3g" % (e_opt.max(), np.quantile(e_samp, 0.99), e_samp.max()))
    assert e_opt.max() <= STATE_FP64_P99
    assert np.quantile(e_samp, 0.99) <= STATE_FP64_P99 and e_samp.max() <= STATE_FP64_MAX
    ctrl.set_sampled_top_n(9)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        _, _, opt2, samp2 = ctrl._calc_input_control(X0)
    assert samp2.shape == (9, T, 3) and opt2.shape == (T, 3) and np.count_nonzero(samp2) > 0.9 * samp2.size
    assert np.all(np.diff(ctrl.last_top_cost) >= 0)


def test_viewer_calls_leave_the_next_tick_unchanged():
    K, T = 50000, 12
    g = Golden("diffdrive_pe0.05")
    sp = _spec(K, T, _mlp(3, 2))
    out = []
    for view in (False, True):
        eng = _engine(sp, g.path)
        eng.set_keep_costs(True)
        eng.set_nominal(np.random.default_rng(2).normal(0, 0.5, (T, 2)).astype(np.float32))
        eng.step(X0, None, seed=3, tick=1)
        if view:
            X = torch.zeros(K, T, 3, dtype=torch.float32, device="cuda")
            eng.trajectories(X0, X, True, None, seed=3, tick=1)
            top = torch.zeros(K // 10, T, 3, dtype=torch.float32, device="cuda")
            eng.top_trajectories(X0, top, K // 10, want_optimal=True, index_shift=0, seed=3, tick=1)
        u0, useq = eng.step(X0 + 0.05, None, seed=3, tick=2)
        out.append((u0.copy(), useq.copy(), eng.get_nominal().copy(), eng.get_waypoint_idx()))
        assert eng.check_guards() == 0
        eng.close()
    for a, b in zip(*out):
        assert np.array_equal(a, b)


def test_viewer_refusals_keep_their_status_codes():
    from mppi_b200 import _lib
    g = Golden("diffdrive_pe0.05")
    K, T = 256, 12
    sp = _spec(K, T, _mlp(3, 2))
    eng = _engine(sp, g.path)
    eng.step(X0, None, seed=3, tick=1)
    lib, x0 = eng.lib, X0.ctypes.data_as(_lib._PD)
    traj = torch.zeros(K + 1, T, 3, dtype=torch.float32, device="cuda")
    top = lambda n: lib.mppi_get_top_trajectories(eng._h, x0, None, 3, 1, n, 1, None, _fptr(traj), None, None)  # noqa: E731
    assert top(4) == MPPI_E_STATE                              # keep_costs is off
    eng.set_keep_costs(True)
    eng.step(X0, None, seed=3, tick=1)
    assert top(0) == MPPI_E_BADARG and top(K + 1) == MPPI_E_BADARG
    assert top(K) == 0
    eng.close()
    fleet = engine_from_spec(orc.diffdrive_spec(K=K, T=T, cost_mode="sum", waypoint_mode="frozen"), g.path, n_robots=2)
    assert fleet.lib.mppi_get_trajectories(fleet._h, x0, None, 3, 1, None, _fptr(traj)) == MPPI_E_UNSUPPORTED
    fleet.close()
