"""Cost of per-robot scenes: the same fleet tick with the shared obstacle set (constant-bank operands) and with every robot's own
set (mppi_set_robot_obstacles: shared-memory operands loaded in the prologue), alternated in one process.  Device time per tick
(CUDA events; open loop: around back-to-back ticks after a warm-up; closed loop: whole calls of two lengths, differenced), for 4096 diff-drive robots x K = 1024 x
T = 30 with 8 circles each (same circles in both arms, so the sample costs and the work are the same), plus the race-car
fleet with footprint obstacles.  Prints the GPU name and power limit with the numbers; `--json PATH` also writes them there."""
import json
import os
import subprocess
import sys

sys.path[:0] = [os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", d) for d in (".", "dnn-mppi-mpc_b200", "tests")]
import numpy as np  # noqa: E402
import torch  # noqa: E402
from golden_util import Golden  # noqa: E402
from mppi_b200.batched import BatchedMPPI  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:                                  # noqa: BLE001 -- informational only
        q = torch.cuda.get_device_name(0)
    return q


def make(kind, R, K, T, per_robot):
    if kind == "diffdrive":
        path = Golden("diffdrive_pe0.05").path
        obs = np.array([[path[i, 0] + 0.3, path[i, 1], 0.4] for i in range(10, 170, 20)], dtype=np.float32).astype(np.float64)
        b = BatchedMPPI(R, path, num_samples_K=K, num_horizons_T=T, temperature=2.0, obstacle_circles=obs, margin=1.2, seed=3)
        x0 = np.stack([np.append(path[r % 160, :2], path[r % 160, 2]) for r in range(R)])
    else:
        path = Golden("racecar_noobs").path
        obs = np.array([[path[i, 0], path[i, 1] + 1.0, 0.8] for i in range(5, 85, 10)], dtype=np.float32).astype(np.float64)
        b = BatchedMPPI(R, path, model="bicycle", delta_t=0.05, max_u=(0.523, 2.0), num_samples_K=K, num_horizons_T=T,
                        param_exploration=0.01, param_lambda=50.0, param_alpha=1.0, sigma=((0.5, 0.0), (0.0, 0.1)),
                        stage_cost_weight=(50.0, 50.0, 1.0, 20.0), terminal_cost_weight=(50.0, 50.0, 1.0, 20.0),
                        window=200, obstacle_circles=obs, margin=1.5, seed=3)
        x0 = np.stack([path[r % 90] for r in range(R)])
    if per_robot:
        b.set_obstacles(np.tile(obs[None], (R, 1, 1)))
    return b, torch.from_numpy(x0.astype(np.float32)).cuda().contiguous(), x0


def open_loop_ms(b, x0_d, n=40, warm=10):
    for _ in range(warm):
        b.step(x0_d)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        b.step(x0_d)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def closed_loop_ms(b, x0, n_short=10, n_long=40):
    """Device time per closed-loop tick: CUDA events around a whole call (state upload, one graph of n launches, log
    download) for n_long and n_short ticks; the difference over n_long - n_short leaves the per-call copies out."""
    def call_ms(n):
        b.run_closed_loop(x0, n)                       # first call of this length instantiates its graph
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()                                    # the fleet runs on torch's current stream
        b.run_closed_loop(x0, n)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    return (call_ms(n_long) - call_ms(n_short)) / (n_long - n_short)


def main():
    info = gpu_info()
    print("GPU:", info)
    out = {"gpu": info, "rows": []}
    for kind, R, K, T in (("diffdrive", 4096, 1024, 30), ("bicycle", 512, 1024, 50)):
        res = {"shared": [], "per_robot": [], "shared_closed": [], "per_robot_closed": []}
        for rep in range(3):                           # alternate the two arms
            for per_robot in (False, True):
                b, x0_d, x0 = make(kind, R, K, T, per_robot)
                arm = "per_robot" if per_robot else "shared"
                res[arm].append(open_loop_ms(b, x0_d))
                res[arm + "_closed"].append(closed_loop_ms(b, x0))
                b.engine.close()
        row = {"fleet": kind, "R": R, "K": K, "T": T}
        for k, v in res.items():
            row[k + "_ms"] = float(np.median(v))
            row[k + "_all_ms"] = [round(x, 4) for x in v]
        row["open_loop_ratio"] = row["per_robot_ms"] / row["shared_ms"]
        row["closed_loop_ratio"] = row["per_robot_closed_ms"] / row["shared_closed_ms"]
        out["rows"].append(row)
        print("%-9s R=%d K=%d T=%d  open loop: shared %.4f ms, per-robot %.4f ms (x%.3f)  closed loop: shared %.4f ms, "
              "per-robot %.4f ms (x%.3f) per tick" % (kind, R, K, T, row["shared_ms"], row["per_robot_ms"], row["open_loop_ratio"],
                                                      row["shared_closed_ms"], row["per_robot_closed_ms"], row["closed_loop_ratio"]))
    if "--json" in sys.argv:
        with open(sys.argv[sys.argv.index("--json") + 1], "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
