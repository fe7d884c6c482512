"""The drop-in boundary (SURVEY.md 8b): every host class keeps the reference class's constructor parameters (names,
order, defaults) and per-tick method name.  The expected signatures below were read off the reference sources
(file:line cited per entry)."""
import inspect

import pytest

# (module, class, tick method, reference file:line, positional parameters in order, defaults of the trailing ones)
EXPECTED = [
    ("mppi_b200.mppi_differential_drive", "MPPIAlgorithms", "_calc_input_control",
     "controllers/mppi_differential_drive.py:44-60",
     ["delta_t", "ref_path", "max_speed", "max_omega", "num_samples_K", "num_horizons_T", "param_exploration",
      "param_lambda", "param_alpha", "sigma", "stage_cost_weight", "terminal_cost_weight", "visualize_optimal_traj",
      "visualze_sampled_trajs"], {"visualize_optimal_traj": True, "visualze_sampled_trajs": True}),
    ("mppi_b200.mppi_differential_drive_obs", "MPPIAlgorithms", "_calc_input_control",
     "controllers/mppi_differential_drive_obs.py:44-62",
     ["delta_t", "ref_path", "max_speed", "max_omega", "num_samples_K", "num_horizons_T", "param_exploration",
      "param_lambda", "param_alpha", "sigma", "stage_cost_weight", "terminal_cost_weight", "obstacle_circles",
      "safety_margin_rate", "visualize_optimal_traj", "visualze_sampled_trajs"],
     {"visualize_optimal_traj": True, "visualze_sampled_trajs": True}),
    ("mppi_b200.mppi_differential_drive_goal", "MPPIAlgorithms", "_calc_input_control",
     "test/mppi_differential_drive_obs.py:44-62",
     ["delta_t", "goal_point", "max_speed", "max_omega", "num_samples_K", "num_horizons_T", "param_exploration",
      "param_lambda", "param_alpha", "sigma", "stage_cost_weight", "terminal_cost_weight", "obstacle_circles",
      "safety_margin_rate", "visualize_optimal_traj", "visualze_sampled_trajs"],
     {"visualize_optimal_traj": True, "visualze_sampled_trajs": True}),
    ("mppi_b200.mppi_race_car_obstacle", "MPPIRacecarController", "_calc_control_input",
     "controllers/mppi_race_car_obstacle.py:11-30",
     ["delta_t", "wheel_base", "max_steer_abs", "max_accel_abs", "ref_path", "horizon_step_T", "number_of_samples_K",
      "param_exploration", "param_lambda", "param_alpha", "sigma", "stage_cost_weight", "terminal_cost_weight",
      "obstacle_circles", "collision_safety_margin_rat", "visualize_optimal_traj", "visualze_sampled_trajs"],
     {"delta_t": 0.05, "wheel_base": 2.5, "max_steer_abs": 0.523, "max_accel_abs": 2.0, "horizon_step_T": 10,
      "number_of_samples_K": 100, "param_exploration": 0.01, "param_lambda": 50.0, "param_alpha": 1.0,
      "collision_safety_margin_rat": 1.5}),
]
# the first positional parameter that has a default in the reference: it and every later one may be omitted by a caller
# (in the race-car class that includes the array-valued ref_path, sigma, weights and obstacle_circles, :11-30)
FIRST_DEFAULTED = {"mppi_b200.mppi_differential_drive": "visualize_optimal_traj",
                   "mppi_b200.mppi_differential_drive_obs": "visualize_optimal_traj",
                   "mppi_b200.mppi_differential_drive_goal": "visualize_optimal_traj",
                   "mppi_b200.mppi_race_car_obstacle": "delta_t"}


def _positional(cls):
    sig = inspect.signature(cls.__init__)
    ps = [p for p in list(sig.parameters.values())[1:] if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
    return [p.name for p in ps], {p.name: p.default for p in ps if p.default is not p.empty}


@pytest.mark.parametrize("mod,cls,tick,ref,names,defaults", EXPECTED, ids=[e[0].split(".")[-1] for e in EXPECTED])
def test_drop_in_signature_matches_the_reference_source(mod, cls, tick, ref, names, defaults):
    import importlib
    c = getattr(importlib.import_module(mod), cls)
    got_names, got_defaults = _positional(c)
    assert got_names == names, ref
    for k, v in defaults.items():
        assert got_defaults[k] == v, (ref, k)
    assert [n for n in got_names if n in got_defaults] == names[names.index(FIRST_DEFAULTED[mod]):], ref
    assert callable(getattr(c, tick))
    # everything this repo adds is keyword-only, so positional call sites of the reference keep working
    params = inspect.signature(c.__init__).parameters.values()
    extra = {p.name for p in params if p.kind is p.KEYWORD_ONLY}
    forwards = any(p.kind is p.VAR_KEYWORD for p in params)           # subclasses forward **kw to the base class
    assert {"seed", "device"} <= extra or forwards
