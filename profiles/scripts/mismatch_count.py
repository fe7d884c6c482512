"""K=1M, H=50 diff-drive (sum/frozen, Philox): how many samples' costs differ from the FP64 C oracle by more than
rtol 1e-5 (= nearest-waypoint near-ties decided differently in FP32), for the library MPPI_B200_LIB points at.
Test infrastructure use of oracle/ (same check as tests/test_gpu_parity.py::test_large_K_full_size_property)."""
import os, sys; sys.path[:0] = [os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np, torch
from golden_util import Golden
from gpu_util import engine_from_spec
from oracle import c_oracle as co, mppi_oracle as orc
g = Golden("diffdrive_pe0.05")
K, T = 1 << 20, 50
sp = orc.diffdrive_spec(K=K, T=T, param_exploration=0.05, param_lambda=1.0, cost_mode="sum", waypoint_mode="frozen")
sp.temperature = 5.0
eng = engine_from_spec(sp, g.path)
for x0, seed in ((np.array([0.5, 0.6, 0.7]), 2024), (np.array([2.9, 2.2, 1.2]), 7)):
    eps = torch.zeros(K, T, 2, dtype=torch.float32, device="cuda")
    eng.generate_noise(eps, seed=seed, tick=3)
    S = torch.zeros(K, dtype=torch.float32, device="cuda")
    eng.set_waypoint_idx(0)
    eng.rollout_costs(x0, S, None, seed=seed, tick=3)
    eps_h = eps.cpu().numpy()
    So, _, _ = co.costs(sp, g.path, np.zeros((T, 2)), 0, x0, eps_h)
    Sg = S.cpu().numpy()
    bad = np.nonzero(np.abs(Sg - So) > 1e-6 + 1e-5 * np.abs(So))[0]
    wp_m = orc.decision_margins(sp, g.path, np.zeros((T, 2)), 0, x0, eps_h[bad])[0] if bad.size else np.zeros(1)
    print(f"x0={x0} mismatching samples {bad.size} of {K} ({bad.size / K:.2e}); worst FP64 decision margin among them {wp_m.max():.2e}")
