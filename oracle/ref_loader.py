"""TEST INFRASTRUCTURE ONLY -- loads the *unmodified* reference controllers from
/root/reference so the oracle restatement (oracle/mppi_oracle.py, oracle/mppi_oracle.c)
can be pinned against them and golden vectors can be generated.

/root/reference exists only in the build container, never on the GPU box, so nothing
that runs under `-m gpu`, `smoke()` or `bench.py` may import this module.  It is used
only by `tests/golden/make_golden.py` (the fixture generator); the tests read what it stored.

The reference imports matplotlib at module top
(controllers/mppi_differential_drive.py:6,8; models/vehicle.py:2-5) but only uses it
inside plotting code the harness never calls, so stub modules are enough.
"""
import os
import sys
import types
import io
import contextlib

import numpy as np

REFERENCE_ROOT = os.environ.get("MPPI_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "controllers"))


class _Stub(types.ModuleType):
    def __getattr__(self, k):
        if k.startswith("__"):
            raise AttributeError(k)
        return _Stub(k)

    def __call__(self, *a, **kw):
        return _Stub("x")


_loaded = {}


def load_reference():
    """Returns a dict of the reference classes / helpers, importing them once."""
    if _loaded:
        return _loaded
    if not reference_available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    for n in ("matplotlib", "matplotlib.pyplot", "matplotlib.animation",
              "matplotlib.patches", "matplotlib.collections"):
        sys.modules.setdefault(n, _Stub(n))
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    from controllers.mppi_differential_drive import MPPIAlgorithms, DifferentialDrive
    from controllers.mppi_differential_drive_obs import MPPIAlgorithms as MPPIObs
    from controllers.mppi_race_car_obstacle import MPPIRacecarController
    from controllers.mppi_race_car import MPPIRacecarController as MPPIRacecarNoObs
    from path_generator.cubic_spline_planner import calc_spline_course
    _loaded.update(dict(
        MPPIAlgorithms=MPPIAlgorithms, DifferentialDrive=DifferentialDrive,
        MPPIObs=MPPIObs, MPPIRacecarController=MPPIRacecarController,
        MPPIRacecarNoObs=MPPIRacecarNoObs, calc_spline_course=calc_spline_course))
    return _loaded


def load_reference_extras():
    """The two MPPI scripts under the reference's test/ directory that SURVEY.md 8f row 3 names:
      * test/mppi_differential_drive_obs.py -- the goal-point diff-drive MPPI class (in-repo numpy loops);
      * test/test_mppi_diff_obs.py -- `dynamics`, `running_cost` (moving soft obstacles) and the
        `MPPIWrapper._compute_rollout_costs` loop.  That script subclasses pytorch_mppi.MPPI, a package that is
        neither vendored nor pinned by the reference; a bare stand-in class lets the module import so its OWN
        functions can be executed -- the pytorch_mppi update rule itself stays unavailable (parity unpinned)."""
    if "GoalMPPI" in _loaded:
        return _loaded
    load_reference()
    import importlib
    pm = types.ModuleType("pytorch_mppi")

    class MPPI:                                    # stand-in base class, never instantiated
        pass
    pm.MPPI = MPPI
    sys.modules.setdefault("pytorch_mppi", pm)
    goal_mod = importlib.import_module("test.mppi_differential_drive_obs")
    dyn_mod = importlib.import_module("test.test_mppi_diff_obs")
    _loaded.update(dict(GoalMPPI=goal_mod.MPPIAlgorithms, GoalPlant=goal_mod.DifferentialDrive,
                        dynobs_dynamics=dyn_mod.dynamics, dynobs_running_cost=dyn_mod.running_cost,
                        dynobs_wrapper=dyn_mod.MPPIWrapper,
                        dynobs_positions=dyn_mod.initial_obstacle_positions.numpy().copy(),
                        dynobs_velocities=dyn_mod.obstacle_velocities.numpy().copy()))
    return _loaded


def load_reference_mlps():
    """The reference's residual-MLP torch modules: dnn/simple_mlp.py:MultiLayerPerception (3 inputs) and the
    5-input MultiLayerPerceptron of simulation/bullet_differential_drive_dnn.py:37-60 (that script imports casadi,
    pybullet, l4casadi, torchvision and acados at module top; none is touched by the class, stubs are enough)."""
    if "MLP3" in _loaded:
        return _loaded
    load_reference()
    import importlib
    for n in ("casadi", "pybullet", "pybullet_data", "l4casadi", "torchvision", "torchvision.models", "acados_template"):
        sys.modules.setdefault(n, _Stub(n))
    m3 = importlib.import_module("dnn.simple_mlp")
    m5 = importlib.import_module("simulation.bullet_differential_drive_dnn")
    # the three-hidden-layer class the *_3l*.pth checkpoints were trained with (train/train_diff_mlp.py:13-36)
    m5l3 = importlib.import_module("train.train_diff_mlp")
    _loaded.update(dict(MLP3=m3.MultiLayerPerception, MLP5=m5.MultiLayerPerceptron, MLP5_3L=m5l3.MultiLayerPerceptron))
    return _loaded


def instrument(ctrl, eps_list):
    """Make a reference controller deterministic and observable without editing it.

    * `_calc_epsilon` (the only RNG use: mppi_differential_drive.py:282,
      mppi_race_car_obstacle.py:144) is replaced by a pop from `eps_list`.
    * `_compute_weight` is wrapped to capture S and w; `_moving_average_filter` to
      capture the raw and filtered weighted-noise sum.
    Returns the dict the captures land in (overwritten every tick).
    """
    cap = {}
    it = iter(eps_list)
    ctrl._calc_epsilon = lambda *a, **k: next(it).copy()
    _w = ctrl._compute_weight

    def cw(S):
        cap["S"] = np.array(S, copy=True)
        w = _w(S)
        cap["w"] = np.array(w, copy=True)
        return w
    ctrl._compute_weight = cw
    _f = ctrl._moving_average_filter

    def mf(xx, window_size):
        cap["w_eps"] = np.array(xx, copy=True)
        out = _f(xx, window_size)
        cap["w_eps_filt"] = np.array(out, copy=True)
        return out
    ctrl._moving_average_filter = mf
    return cap


@contextlib.contextmanager
def quiet():
    """The reference prints '[ERROR] Reached the end ...' at path end; swallow stdout."""
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        yield buf
