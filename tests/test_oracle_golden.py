"""Pins the oracle (test infrastructure) to the golden vectors produced by the unmodified
reference classes: scalar-loop restatement bit-exact, vectorised and C restatements to
1e-12 (diff-drive, FP64) / 4e-6 (race-car: the reference accumulates in FP32)."""
import os

import numpy as np
import pytest

from golden_util import ALL_CASES, DIFFDRIVE_CASES, RACECAR_CASES, Golden, rel_err
from oracle import c_oracle as co
from oracle import mppi_oracle as orc


def _degenerate(g, i):
    """Every sample collided: S - rho has no tracking-cost bits left in the FP32 reference
    (ulp(1e10) = 1024), so weights are rounding noise there (SURVEY.md section 7)."""
    return g.rec["S"][i].min() >= 1e10 and g.rec["S"][i].dtype == np.float32


@pytest.mark.parametrize("name", ALL_CASES)
def test_loops_restatement_is_bit_exact(name):
    g = Golden(name)
    sp = g.spec()
    for i in range(min(g.n_ticks, 2)):
        o = orc.tick_loops(sp, **g.tick_inputs(i))
        for k in ("S", "w", "w_eps", "w_eps_filt", "U_after", "u0"):
            assert np.array_equal(np.asarray(o[k]), g.rec[k][i]), (name, i, k)
        assert o["idx_after"] == g.rec["idx_after"][i]


@pytest.mark.parametrize("name", ALL_CASES)
def test_vectorised_restatement(name):
    g = Golden(name)
    sp = g.spec()
    f32 = name in RACECAR_CASES
    for i in range(g.n_ticks):
        o = orc.tick_vec(sp, **g.tick_inputs(i))
        assert rel_err(o["S"], g.rec["S"][i]) <= (1e-6 if f32 else 1e-12)
        assert o["idx_after"] == g.rec["idx_after"][i]
        if _degenerate(g, i):
            continue
        tol = 2e-6 if f32 else 1e-12
        assert np.max(np.abs(o["w"] - g.rec["w"][i])) <= tol
        assert np.max(np.abs(o["U_after"] - g.rec["U_after"][i])) <= tol
        assert np.max(np.abs(o["u0"] - g.rec["u0"][i])) <= tol


@pytest.mark.parametrize("name", ALL_CASES)
def test_c_restatement(name):
    g = Golden(name)
    sp = g.spec()
    f32 = name in RACECAR_CASES
    for i in range(g.n_ticks):
        o = co.tick(sp, **g.tick_inputs(i))
        assert rel_err(o["S"], g.rec["S"][i]) <= (4e-6 if f32 else 1e-12)
        assert o["idx_after"] == g.rec["idx_after"][i]
        if _degenerate(g, i):
            continue
        tol = 2e-5 if f32 else 1e-12
        assert np.max(np.abs(o["w_eps"] - g.rec["w_eps"][i])) <= tol
        assert np.max(np.abs(o["U_after"] - g.rec["U_after"][i])) <= tol


def test_closed_loop_trace_reproduced_by_oracle():
    """40-tick closed loop (plant = DifferentialDrive.update_state): drive the C oracle with its
    OWN outputs and land on the reference's trajectory."""
    g = Golden("diffdrive_closed_loop")
    sp = g.spec()
    x = g.rec["x0"][0].copy()
    U = g.rec["U0"][0].copy()
    idx = int(g.rec["idx0"][0])
    for i in range(g.n_ticks):
        assert np.max(np.abs(x - g.rec["x0"][i])) < 1e-9
        o = co.tick(sp, g.path, U, idx, x, g.eps[i])
        U, idx = o["U_after"], o["idx_after"]
        x = orc.plant_diffdrive(x, o["u0"], sp.dt)
    assert idx == g.rec["idx_after"][-1]


@pytest.mark.parametrize("kind", ["diffdrive", "racecar"])
@pytest.mark.parametrize("T", [10, 12, 20, 30, 50])
def test_filter_matrices(kind, T):
    import os
    from golden_util import GOLDEN_DIR
    M = np.load(os.path.join(GOLDEN_DIR, "filter_matrices.npz"))["%s_T%d" % (kind, T)]
    assert np.max(np.abs(orc.filter_matrix(T, kind) - M)) == 0.0
    assert np.max(np.abs(co.filter_matrix(T, kind) - M)) < 1e-8
    if kind == "diffdrive":            # the tail bug (Q7): last row gain 3.307, row sum ~1.98
        assert abs(M[-1].sum() - 0.6 * (10 / 6) * (10 / 7) * (10 / 8) * (10 / 9)) < 1e-12
    else:
        assert np.allclose(M.sum(axis=1), 1.0, atol=1e-6)


def test_frozen_and_sum_modes_agree_between_evaluators():
    """The non-literal mode combinations (perf modes) have no reference class; the three
    restatements must still agree with each other."""
    g = Golden("diffdrive_pe0.05")
    for cm in ("last", "sum"):
        for wm in ("strict", "frozen"):
            sp = g.spec(cost_mode=cm, waypoint_mode=wm)
            inp = g.tick_inputs(1)
            a = orc.tick_loops(sp, **inp)
            b = orc.tick_vec(sp, **inp)
            c = co.tick(sp, **inp)
            assert rel_err(b["S"], a["S"]) < 1e-12 and rel_err(c["S"], a["S"]) < 1e-12
            assert a["idx_after"] == b["idx_after"] == c["idx_after"]
            assert np.max(np.abs(c["U_after"] - a["U_after"])) < 1e-12


def test_philox_known_answers():
    """Random123 known-answer vectors for Philox4x32-10."""
    kat = [([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
           ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
           ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
            [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]
    for ctr, key, out in kat:
        assert list(co.philox(ctr, key)) == out
        assert list(orc.philox4x32(np.array(ctr, np.uint32), np.array(key, np.uint32))) == out


def test_philox_noise_statistics_and_c_agreement():
    sigma = np.array([[0.1, 0.02], [0.02, 0.05]])
    e = orc.philox_noise(seed=1234, tick=3, K=20000, T=7, sigma=sigma)
    flat = e.reshape(-1, 2)
    assert np.all(np.abs(flat.mean(0)) < 5e-3)
    assert np.max(np.abs(np.cov(flat.T) - sigma)) < 3e-3
    # C oracle in Philox mode == Python Philox noise injected
    g = Golden("diffdrive_pe0.05")
    sp = g.spec(waypoint_mode="frozen", cost_mode="sum")
    inp = g.tick_inputs(2)
    eps = orc.philox_noise(7, 5, sp.K, sp.T, sp.sigma)
    a = co.tick(sp, inp["path"], inp["U"], inp["idx"], inp["x0"], eps=None, seed=7, tick=5)
    b = co.tick(sp, inp["path"], inp["U"], inp["idx"], inp["x0"], eps=eps.astype(np.float32))
    assert rel_err(a["S"], b["S"]) < 1e-5


@pytest.mark.parametrize("name", ["diffdrive_viz", "racecar_viz"])
def test_visualisation_outputs_and_nominal_clamp(name):
    """A16 / Q9: with the visualisation flags on, the reference replays the updated nominal and every sample
    with t-1 indexing and clamps the stored nominal in place; the loop restatement is bit-exact."""
    g = Golden(name)
    sp = g.spec()
    for i in range(g.n_ticks):
        o = orc.tick_loops(sp, **g.tick_inputs(i))
        assert np.array_equal(o["U_after"], g.rec["U_after"][i])
        assert np.array_equal(o["optimal_traj"], g.rec["optimal_traj"][i])
        assert np.array_equal(o["sampled_traj"], g.rec["sampled_traj"][i])
    lim = np.asarray(sp.u_max)
    assert np.all(np.abs(g.rec["U_after"]) <= lim + 1e-6) and np.any(np.abs(g.rec["U_after"]) >= lim - 1e-6)


def test_target_soft_running_cost_matches_reference_functions():
    """SURVEY 8f row 3: the moving-soft-obstacle running cost.  The golden S is what the reference's own
    `dynamics` + `running_cost` produce inside its `MPPIWrapper._compute_rollout_costs` loop
    (test/test_mppi_diff_obs.py:28-66,113-151, float32 torch) for the stored clamped controls; the three
    restatements must reproduce it (FP32 summation over 25 steps: 2e-6 relative)."""
    from golden_util import TARGET_SOFT_CASE
    g = Golden(TARGET_SOFT_CASE)
    sp = g.spec()
    for i in range(g.n_ticks):
        inp = g.tick_inputs(i)
        V, _ = orc.rollout_states(sp, np.asarray(inp["U"], np.float32), np.asarray(inp["x0"], np.float32), inp["eps"])
        assert np.array_equal(V, g.rec["V"][i])                      # same clamped controls as the harness fed
        S_vec, _, _ = orc.costs_vec(sp, None, inp["U"], 0, inp["x0"], inp["eps"])
        assert rel_err(S_vec, g.rec["S"][i]) <= 2e-6, i
        S_c, _, _ = co.costs(sp, None, inp["U"], 0, inp["x0"], inp["eps"])
        assert rel_err(S_c, g.rec["S"][i]) <= 2e-6, i
    sp_small = g.spec(K=24)
    inp = g.tick_inputs(0)
    a = orc.tick_loops(sp_small, None, inp["U"], 0, inp["x0"], inp["eps"][:24])
    assert rel_err(a["S"], g.rec["S"][0][:24]) <= 2e-6


@pytest.mark.parametrize("n_in,n_hidden", [(3, 2), (5, 2), (5, 3)])
def test_mlp_forward_matches_reference_torch_modules(n_in, n_hidden):
    """SURVEY 8f row 4: the oracle's residual MLP vs forward passes of the reference's own torch modules
    (tests/golden/mlp_forward.npz), including the StandardScaler pre/post-processing of the 5-input model."""
    import os
    from golden_util import GOLDEN_DIR
    z = np.load(os.path.join(GOLDEN_DIR, "mlp_forward.npz"))
    w = orc.make_mlp(seed=5, out_scale=0.01, dtype=np.float64, n_in=n_in, scalers=(n_in == 5), n_hidden=n_hidden)
    tag = "%d" % n_in + ("_3l" if n_hidden == 3 else "")       # 5_3l: the class of train/train_diff_mlp.py:13-36
    X = z["X" + tag]
    y = orc.mlp_forward(w, X[:, :3], X[:, 3:] if n_in == 5 else None)
    assert np.max(np.abs(y - z["Y" + tag])) <= 1e-12


@pytest.mark.parametrize("ckpt,scalers,cls_key", [("mlp_diff_300x100.pth", "scalers_mlp_diff_300x100_20_l.pth", "MLP5"),
                                                  ("mlp_diff_300x100_3l_mppi.pth", "scalers_mlp_diff_300x100_3l_mppi.pth", "MLP5_3L")])
def test_oracle_mlp_matches_the_trained_reference_model(ckpt, scalers, cls_key):
    """The TRAINED residuals (saved_models/mlp_diff_300x100*.pth + their scalers; the *_3l one has three hidden layers,
    train/train_diff_mlp.py:13-36) vs the oracle restatement.  tests/golden/trained_<checkpoint>.npz holds the checkpoint's
    weights verbatim, its StandardScaler statistics and forward passes of the reference's own torch class with the sklearn
    scalers applied (make_golden.py trained) on 64 inputs."""
    import json
    from golden_util import GOLDEN_DIR
    z = np.load(os.path.join(GOLDEN_DIR, "trained_%s.npz" % ckpt[:-len(".pth")]))
    meta = json.loads(str(z["meta"]))
    assert meta["checkpoint"] == "saved_models/" + ckpt and meta["scalers"] == "saved_models/" + scalers
    n_hidden = 3 if cls_key == "MLP5_3L" else 2
    assert meta["n_hidden"] == n_hidden
    w = {k: z[k].astype(np.float64) for k in z.files if k not in ("meta", "X", "Y_ref")}
    assert sorted(k for k in w if k[0] == "W") == ["W%d" % i for i in range(n_hidden + 2)]
    X, y_ref = z["X"], z["Y_ref"]
    y = orc.mlp_forward(w, X[:, :3], X[:, 3:])
    assert np.max(np.abs(y - y_ref)) <= 1e-10 * max(1.0, np.max(np.abs(y_ref)))


def test_spline_course_restatement_is_bit_exact():
    """SURVEY 8f row 4: calc_spline_course (path_generator/cubic_spline_planner.py:311-323) restated in
    oracle/spline_oracle.py vs courses produced by the unmodified reference function."""
    import json
    from golden_util import GOLDEN_DIR
    from oracle.spline_oracle import spline_course
    g = np.load(os.path.join(GOLDEN_DIR, "paths.npz"))["spline"]
    c = spline_course([0.0, 0.5, 1.0, 3.0, 3.0, 1.0, -4.0], [0.0, 1.0, 1.0, 2.0, 5.0, 1.0, -1.0], 0.1)
    assert np.array_equal(c, g)
    z = np.load(os.path.join(GOLDEN_DIR, "spline_courses.npz"))
    for i, case in enumerate(json.loads(str(z["meta"]))["cases"]):
        c = spline_course(z["wx%d" % i], z["wy%d" % i], case["ds"])
        assert c.shape == (case["n_pts"], 3) and np.array_equal(c, z["course%d" % i]), i
