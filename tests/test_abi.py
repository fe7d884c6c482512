"""CPU checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every
symbol include/mppi_b200.h declares; handle creation fails loudly (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "mppi_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mppi_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported_and_bound():
    from mppi_b200 import _lib
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), "libmppi_b200.so does not export %s" % n
        assert n in _lib.SYMBOLS, "ctypes binding table misses %s" % n
    assert sorted(_lib.SYMBOLS) == names
    assert lib.mppi_abi_version() == _lib.MPPI_ABI_VERSION == 3


def test_config_struct_layout_matches_header():
    from mppi_b200 import _lib
    # 16 int32 + 32 doubles, naturally aligned
    assert C.sizeof(_lib.MppiConfig) == 16 * 4 + 32 * 8
    c = _lib.MppiConfig()
    _lib.load().mppi_default_config(C.byref(c))
    assert (c.abi_version, c.K, c.T, c.window, c.n_robots, c.cost_kind) == (3, 1000, 30, 20, 1, 0)
    assert abs(c.dt - 0.1) < 1e-15 and abs(c.sigma[3] - 0.01) < 1e-15 and c.vehicle_l == 4.0
    assert c.soft_obs_weight == 100.0 and c.soft_obs_safety == 2.0 and c.ctrl_w[1] == 0.1      # trailing fields line up


def test_errors_are_status_codes_not_exceptions_across_the_abi():
    from mppi_b200 import _lib
    lib = _lib.load()
    assert lib.mppi_create(None, None) == -1
    assert lib.mppi_destroy(None) == -1
    assert b"invalid" in lib.mppi_strerror(-1)
    c = _lib.MppiConfig()
    lib.mppi_default_config(C.byref(c))
    c.T = 4                                     # the reference filter raises for T < 10 (:263)
    h = C.c_void_p()
    assert lib.mppi_create(C.byref(c), C.byref(h)) == -1 and not h.value


def test_no_cpu_fallback():
    """Without a CUDA device the drop-in class refuses to construct.  Checked in a child process that sees no device, so
    the check also runs on a machine that has one."""
    import subprocess
    import sys
    code = ("import sys\n"
            "sys.path.insert(0, %r)\n"
            "import numpy as np\n"
            "from mppi_b200 import MppiError\n"
            "from mppi_b200.mppi_differential_drive import MPPIAlgorithms\n"
            "try:\n"
            "    MPPIAlgorithms(0.1, np.zeros((30, 3)), 5.0, 3.14, 100, 10, 1e-4, 1.0, 0.2, np.diag([0.1, 0.01]),\n"
            "                   np.ones(3), np.ones(3))\n"
            "except MppiError:\n"
            "    sys.exit(0)\n"
            "sys.exit('constructed without a CUDA device')\n") % os.path.join(ROOT, "dnn-mppi-mpc_b200")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "dnn-mppi-mpc_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "mppi_oracle" not in txt.replace(
                    "oracle/mppi_oracle.py:philox_noise", ""), f


@pytest.mark.parametrize("n_units,T,n_clusters", [(128, 30, 74), (196, 12, 74), (98, 11, 74), (256, 30, 74), (79, 50, 74),
                                                  (2048, 30, 74), (75, 31, 74), (148, 10, 74)])
def test_mlp_balanced_schedule_is_an_even_partition(n_units, T, n_clusters):
    """Host-side logic of the learned-dynamics kernel's balanced (horizon-split) schedule, through the exported cut
    function the kernel itself evaluates (no GPU): the cluster ranges tile the unit x timestep sequence exactly once, cuts
    fall on even timesteps (a Philox call yields two steps), the load differs by at most a few steps, and whenever the
    launcher's condition holds (n_units * T / n_clusters >= T + 2) a cluster owns at most one tail and one head, the head
    being a different unit from the tail -- what the head-first / tail-last hand-off order relies on."""
    from mppi_b200 import _lib
    lib = _lib.load()
    cuts = [lib.mppi_mlp_schedule_cut(c, n_clusters, n_units, T) for c in range(n_clusters + 1)]
    assert cuts[0] == 0 and cuts[-1] == n_units * T
    assert all(b > a for a, b in zip(cuts, cuts[1:]))
    assert all((c % T) % 2 == 0 for c in cuts[:-1])
    sizes = [b - a for a, b in zip(cuts, cuts[1:])]
    assert max(sizes) - min(sizes) <= 4 and max(sizes) <= n_units * T / n_clusters + 3
    if n_units * T // n_clusters >= T + 2:
        for a, b in zip(cuts, cuts[1:]):
            assert b - a >= T                                   # at least one whole horizon of work
            tail_unit = a // T if a % T else None
            head_unit = (b - 1) // T if b % T else None
            assert tail_unit is None or head_unit is None or head_unit > tail_unit
            # consumer slack: the tail (run last) starts after the producer's head (run first) has finished
            if tail_unit is not None:
                assert (b - a) - (T - a % T) >= a % T
    assert lib.mppi_mlp_schedule_cut(-1, n_clusters, n_units, T) == -1


def test_bench_reference_arm_prints_exactly_one_json_line():
    """bench.py contract: `--impl reference` runs on the host cores only (the oracle port; no GPU, no product code on that
    path) and stdout carries exactly one JSON line with the reference-arm keys."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "sample-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None
