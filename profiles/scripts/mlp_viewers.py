"""Time of the learned-dynamics trajectory viewers at K = 65 536, T = 30 (two and three hidden layers), with CUDA events on
the engine's stream: the top-N replay at n_top = K/10 and the all-K replay (mppi_get_trajectories) per call (see viewer_ms),
and the control tick with the viewers off.  --parent-lib PATH also times the tick of another build of libmppi_b200.so (e.g. the parent commit's), alternating the
two builds process by process (ABBA order) so that both see the same machine state.

    python profiles/scripts/mlp_viewers.py [--parent-lib PATH] [--rounds 6]
"""
import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.join(HERE, "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]

K, T = 65536, 30
X0 = [0.4, 0.3, 0.5]


def _engine(n_hidden):
    from golden_util import Golden
    from gpu_util import engine_from_spec
    from oracle import mppi_oracle as orc
    g = Golden("diffdrive_pe0.05")
    mlp = orc.make_mlp(seed=0, out_scale=0.01, n_hidden=n_hidden)
    sp = orc.diffdrive_spec(K=K, T=T, param_exploration=0.05, cost_mode="sum", waypoint_mode="frozen", model="diffdrive_mlp",
                            mlp=mlp)
    sp.temperature = 2.0
    eng = engine_from_spec(sp, g.path)
    eng.set_mlp([mlp["W%d" % i] for i in range(n_hidden + 2)], [mlp["b%d" % i] for i in range(n_hidden + 2)])
    return eng


def tick_ms(n_hidden, n=50):
    """Control tick, viewers off, on the engine's own stream (events recorded there)."""
    import numpy as np
    import torch
    eng = _engine(n_hidden)
    st = torch.cuda.Stream()
    eng.set_stream(st.cuda_stream)
    x0 = np.array(X0)
    for i in range(5):
        eng.step_async(x0, None, 7, i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for i in range(n):
        eng.step_async(x0, None, 7, 10 + i)
    b.record(st)
    torch.cuda.synchronize()
    eng.close()
    return a.elapsed_time(b) / n


def viewer_ms(n_hidden, n=20):
    """Each viewer call after one tick, on the engine's own stream.  The calls synchronise, so every call is timed on its
    own: `dev` = CUDA events recorded on that stream around the call (sort, control-table kernel, replay kernel and the
    copies, with the launch gaps between them); `wall` = host time of the call, which adds the host synchronisation."""
    import time
    import numpy as np
    import torch
    eng = _engine(n_hidden)
    st = torch.cuda.Stream()
    eng.set_stream(st.cuda_stream)
    eng.set_keep_costs(True)
    x0 = np.array(X0)
    eng.step(x0, None, 7, 0)
    n_top = K // 10
    top = torch.empty(n_top, T, 3, device="cuda")
    allk = torch.empty(K, T, 3, device="cuda")
    torch.cuda.synchronize()
    calls = dict(top=lambda: eng.top_trajectories(x0, top, n_top, want_optimal=True, index_shift=1, seed=7, tick=0),
                 all=lambda: eng.trajectories(x0, allk, True, None, seed=7, tick=0))
    out = {}
    for name, fn in calls.items():
        for _ in range(3):
            fn()
        dev = wall = 0.0
        for _ in range(n):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            t0 = time.perf_counter()
            fn()
            wall += time.perf_counter() - t0
            b.record(st)
            b.synchronize()
            dev += a.elapsed_time(b)
        out[name] = (dev / n, 1e3 * wall / n)
    assert eng.check_guards() == 0
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--tick-only", type=int, default=None, help=argparse.SUPPRESS)     # child process: one tick timing
    args = ap.parse_args()
    if args.tick_only is not None:
        print(json.dumps(dict(tick_ms=tick_ms(args.tick_only))))
        return
    import torch
    name = torch.cuda.get_device_name(0)
    power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip().splitlines()
    print("device: %s, power limit / max SM clock: %s" % (name, power[0] if power else "unknown"))
    for nh in (2, 3):
        v = viewer_ms(nh)
        print("n_hidden=%d K=%d T=%d, per call (device-stream events / host wall): top-N replay (n_top=%d) %.3f / %.3f ms, "
              "all-K replay %.3f / %.3f ms" % (nh, K, T, K // 10, *v["top"], *v["all"]))
    builds = [("this build", None)] + ([("parent build", args.parent_lib)] if args.parent_lib else [])
    for nh in (2, 3):
        res = {b: [] for b, _ in builds}
        for r in range(args.rounds):
            for b, lib in (builds if r % 2 == 0 else builds[::-1]):          # ABBA: neither build always goes first
                env = dict(os.environ)
                if lib:
                    env["MPPI_B200_LIB"] = os.path.abspath(lib)
                out = subprocess.run([sys.executable, __file__, "--tick-only", str(nh)], env=env, capture_output=True, text=True, check=True)
                res[b].append(json.loads(out.stdout.strip().splitlines()[-1])["tick_ms"])
        for b, v in res.items():
            print("n_hidden=%d tick, viewers off, %s: %s ms (median %.4f)" % (nh, b, " ".join("%.4f" % x for x in v), sorted(v)[len(v) // 2]))


if __name__ == "__main__":
    main()
