"""Batched multi-robot mode: R independent differential-drive (or race-car) MPPI controllers solved
in ONE kernel launch (BASELINE config 4).  There is no reference class for this; it is R copies of
the tick of controllers/mppi_differential_drive.py:87-165 (frozen window, per-robot nominal and
waypoint index), each robot drawing its own Philox stream (counter word 3 = robot index).  Besides paths, a fleet can run the
path-free cost kinds (goal point, target pose with moving soft obstacles), and every robot can have its own goal and its own
obstacle set (set_goals / set_obstacles), installed on the device in stream order."""
import numpy as np

from .engine import MPPIEngine


class BatchedMPPI:
    def __init__(self, n_robots, ref_path, *, model="diffdrive", delta_t=0.1, max_u=(5.0, 3.14), num_samples_K=1024,
                 num_horizons_T=30, param_exploration=0.05, param_lambda=1.0, param_alpha=0.2,
                 sigma=((0.1, 0.0), (0.0, 0.01)), stage_cost_weight=(5.0, 5.0, 10.0),
                 terminal_cost_weight=(5.0, 5.0, 10.0), temperature=None, cost_mode="sum", window=20,
                 obstacle_circles=None, margin=1.0, wheel_base=2.5, seed=0, device=0, cost_kind="path", goal=None,
                 collision=None, filter_kind=None, ctrl_w=None, soft_obs_weight=None, soft_obs_safety=None):
        self.R, self.K, self.T = int(n_robots), int(num_samples_K), int(num_horizons_T)
        bicycle = model == "bicycle"
        self.nx = 4 if bicycle else 3
        self.seed = int(seed)
        self._tick = 0
        if collision is None:
            collision = "none" if obstacle_circles is None else ("footprint" if bicycle else "circle")
        if filter_kind is None:
            filter_kind = "racecar" if bicycle else "diffdrive"
        self.cost_kind, self.collision = cost_kind, collision
        self._engine = MPPIEngine(
            model=model, K=self.K, T=self.T, dt=delta_t, u_max=max_u, sigma=np.asarray(sigma, float),
            stage_w=stage_cost_weight, term_w=terminal_cost_weight, param_exploration=param_exploration,
            param_lambda=param_lambda, param_alpha=param_alpha,
            temperature=(param_lambda if bicycle else param_exploration) if temperature is None else temperature,
            window=window, cost_mode=cost_mode, waypoint_mode="frozen",
            filter_kind=filter_kind, yaw_wrap=bicycle, collision=collision,
            obstacles=obstacle_circles, margin=margin, wheel_base=wheel_base, n_robots=self.R, device=device,
            cost_kind=cost_kind, goal=goal, ctrl_w=ctrl_w, soft_obs_weight=soft_obs_weight, soft_obs_safety=soft_obs_safety)
        if ref_path is not None:
            self._engine.set_ref_path(ref_path)
        import torch
        # run on torch's current stream so tensors produced/consumed by torch are naturally ordered
        self._engine.set_stream(torch.cuda.current_stream(device).cuda_stream)
        self._u0 = torch.zeros(self.R, 2, dtype=torch.float32, device="cuda:%d" % device)

    def set_waypoints(self, wx, wy, ds=0.1, max_points=512):
        """One reference path PER ROBOT, generated on the device from (R, n_wp) waypoints by the reference's own course
        generator `calc_spline_course(x, y, ds)` (path_generator/cubic_spline_planner.py:311-323; what the reference
        mains do once on the host, controllers/mppi_differential_drive_cuda.py:400-403).  Accepts numpy arrays or
        CUDA tensors; construct with ref_path=None to start without a shared path."""
        import torch
        dev = "cuda:%d" % self._engine.device
        wx = torch.as_tensor(wx, dtype=torch.float32, device=dev).contiguous()
        wy = torch.as_tensor(wy, dtype=torch.float32, device=dev).contiguous()
        torch.cuda.current_stream(self._engine.device).synchronize()
        self._engine.set_ref_paths_spline(wx, wy, ds, max_points)

    def set_obstacles(self, obs, counts=None):
        """One obstacle set PER ROBOT: (R, m, 3) circles [x, y, r] (circle / footprint collision) or, for the target_soft
        cost kind, (R, m, 4) moving soft obstacles [x, y, vx, vy]; m <= 16.  counts (R,): robot r uses its first counts[r]
        rows.  CUDA tensors are consumed in stream order on the torch stream this fleet runs on (no synchronisation), so
        new obstacles can be computed on the GPU every tick; numpy arrays are uploaded."""
        ncol = 4 if self.cost_kind == "target_soft" else 3
        if len(obs.shape) != 3 or obs.shape[2] != ncol:
            raise ValueError("%s fleet: obstacles are (R, m, %d)" % (self.cost_kind, ncol))
        self._engine.set_robot_obstacles(obs, counts)

    def set_goals(self, goals):
        """One goal PER ROBOT: (R, 2) goal points (cost_kind='goal') or (R, 3) target poses (cost_kind='target_soft'),
        consumed like set_obstacles."""
        self._engine.set_robot_goals(goals)

    def use_shared_scene(self):
        """Every robot scores against the shared goal / obstacles again: the ones given at construction, or the ones last
        installed through engine.set_goal / set_obstacles / set_moving_obstacles."""
        self._engine.use_shared_scene()

    def ref_path(self, robot=0):
        """(N,3) [x, y, yaw] course robot `robot` follows."""
        return self._engine.get_ref_path(robot)[:, :3]

    @property
    def engine(self):
        return self._engine

    def step(self, x0):
        """x0: (R, nx) float32 CUDA tensor.  Returns the (R, 2) float32 CUDA tensor of first controls
        (asynchronous, ordered on the torch stream that was current at construction)."""
        assert x0.is_cuda and tuple(x0.shape) == (self.R, self.nx) and x0.is_contiguous()
        self._engine.step_batched(x0, self._u0, self.seed, self._tick)
        self._tick += 1
        return self._u0

    def run_closed_loop(self, x0, n_ticks):
        """The whole fleet in closed loop ON THE DEVICE: every robot ticks and advances its own plant
        (DifferentialDrive.update_state, controllers/mppi_differential_drive.py:33-40; Vehicle.update for the race-car)
        n_ticks times, no host round trip -- one CUDA graph of n_ticks launches.  x0: (R, nx) array.  Returns
        (states (n+1, R, nx), controls (n, R, 2)) float32."""
        states, controls = self._engine.run_closed_loop(np.asarray(x0, dtype=np.float64), int(n_ticks), self.seed, self._tick,
                                                        1 if self.nx == 4 else 0)
        self._tick += int(n_ticks)
        return states, controls

    def nominal(self):
        self._engine.synchronize()
        return self._engine.get_nominal()

    def waypoint_idx(self):
        self._engine.synchronize()
        return self._engine.get_waypoint_idx()
