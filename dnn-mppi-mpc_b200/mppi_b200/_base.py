"""Shared host logic of the drop-in controller classes (the reference's class surface,
SURVEY.md 8b).  Everything numeric happens behind the C ABI; this file only marshals."""
import warnings

import numpy as np

from .engine import MPPIEngine


def _to_device_noise(noise, K, T, device):
    """Accepts a (K,T,2) numpy array or torch tensor; returns a contiguous float32 CUDA tensor."""
    import torch
    if isinstance(noise, np.ndarray):
        noise = torch.from_numpy(np.ascontiguousarray(noise, dtype=np.float32))
    if tuple(noise.shape) != (K, T, 2):
        raise ValueError("injected noise must have shape (K,T,2) = (%d,%d,2), got %s" % (K, T, tuple(noise.shape)))
    out = noise.to(device="cuda:%d" % device, dtype=torch.float32).contiguous()
    torch.cuda.current_stream(device).synchronize()     # the engine runs on its own stream
    return out


class ControllerBase:
    """Holds one engine handle and mirrors the mutable public state callers touch in the
    reference: `u_prev`, the waypoint index, `ref_path`, `obstacle_circles`."""

    _out_dtype = np.float64
    _idx_attr = "prev_way_point_idx"

    def _init_engine(self, *, ref_path, seed, device, rank, world, **engine_kw):
        self.seed = int(seed)
        self._tick = 0
        self._rank, self._world = int(rank), int(world)
        K_global = engine_kw["K"]
        if world > 1:
            if K_global % world:
                raise ValueError("num_samples_K must be divisible by the world size")
            engine_kw = dict(engine_kw, K=K_global // world, K_global=K_global, k_offset=rank * (K_global // world))
        self._engine = MPPIEngine(device=device, **engine_kw)
        self._K_local = engine_kw["K"]
        self._ref_path = None
        if ref_path is not None:                 # goal / target cost kinds have no reference path
            self.ref_path = ref_path
        self._u_cache = np.zeros((self.T, self.dim_u), dtype=self._out_dtype)
        self._viz_warned = False
        self._top_n = None
        self.last_top_idx = self.last_top_cost = None

    def set_sampled_top_n(self, n_top):
        """Return only the `n_top` lowest-cost sampled trajectories, in ascending cost order, as the 4th element of the
        tick tuple (None restores the reference's (K,T,nx) array).  The reference's viewers draw the samples in
        `np.argsort(S)` order (mppi_differential_drive.py:153) and test/test_mppi_diff_obs.py:102 keeps the top
        max(10, K/10); at K = 1M the full array is 600 MB per tick."""
        self._top_n = None if n_top is None else max(1, min(int(n_top), self._K_local))
        self._engine.set_keep_costs(self._top_n is not None)

    # -- reference attributes ----------------------------------------------------------------
    @property
    def ref_path(self):
        return self._ref_path

    @ref_path.setter
    def ref_path(self, path):
        # re-assigned after construction by the reference main (mppi_race_car_obstacle.py:332)
        self._ref_path = np.asarray(path)
        self._engine.set_ref_path(self._ref_path)

    @property
    def u_prev(self):
        return self._u_cache

    @u_prev.setter
    def u_prev(self, u):
        u = np.asarray(u, dtype=self._out_dtype).reshape(self.T, self.dim_u)
        self._u_cache = u.copy()
        self._engine.set_nominal(u)

    def _get_idx(self):
        return self._engine.get_waypoint_idx()

    def _set_idx(self, v):
        # the reference fails at the next tick on an index outside the path (ValueError from min() / argmin of the empty
        # window slice, mppi_differential_drive.py:214); here the assignment itself is refused
        n = None if self._ref_path is None else len(self._ref_path)
        if n is not None and not (0 <= int(v) < n):
            raise ValueError("waypoint index %d outside the reference path (0..%d)" % (int(v), n - 1))
        self._engine.set_waypoint_idx(int(v))

    # -- one tick ----------------------------------------------------------------------------
    def _tick_impl(self, observed_x, noise=None):
        x = np.asarray(observed_x, dtype=np.float64 if self._out_dtype is np.float64 else np.float32)
        d_eps = None
        if noise is not None:
            d_eps = _to_device_noise(noise, self._K_local, self.T, self._engine.device)
        u0, useq = self._engine.step(x, d_eps, self.seed, self._tick)
        self._tick += 1
        self._u_cache = useq.astype(self._out_dtype)           # returned u aliases u_prev (A2)
        u = self._u_cache
        optimal_traj = np.zeros((self.T, self.dim_x), dtype=self._out_dtype)
        want_opt, want_samp = self._viz_gates()
        if (want_opt or want_samp) and self._top_n:
            import torch
            dev = "cuda:%d" % self._engine.device
            d_samp = torch.empty(self._top_n, self.T, self.dim_x, dtype=torch.float32, device=dev)
            d_idx = torch.empty(self._top_n, dtype=torch.int32, device=dev)
            d_cost = torch.empty(self._top_n, dtype=torch.float32, device=dev)
            opt = self._engine.top_trajectories(x, d_samp, self._top_n, d_idx, d_cost, want_opt, 1, d_eps, self.seed,
                                                self._tick - 1)
            if want_opt:
                optimal_traj = opt.astype(self._out_dtype)
            sampled = d_samp.cpu().numpy().astype(self._out_dtype)
            self.last_top_idx = d_idx.cpu().numpy() + self._rank * self._K_local
            self.last_top_cost = d_cost.cpu().numpy()
        elif (want_opt or want_samp) and self._world == 1:
            import torch
            d_samp = torch.empty(self.K, self.T, self.dim_x, dtype=torch.float32,
                                 device="cuda:%d" % self._engine.device) if want_samp else None
            opt = self._engine.trajectories(x, d_samp, want_opt, d_eps, self.seed, self._tick - 1)
            if want_opt:
                optimal_traj = opt.astype(self._out_dtype)
            sampled = d_samp.cpu().numpy().astype(self._out_dtype) if want_samp else \
                np.broadcast_to(np.zeros((), dtype=self._out_dtype), (self.K, self.T, self.dim_x))
        else:
            # (K,T,nx) zeros like the reference returns when the flag is off, without allocating K*T*nx
            sampled = np.broadcast_to(np.zeros((), dtype=self._out_dtype), (self.K, self.T, self.dim_x))
            if (want_opt or want_samp) and not self._viz_warned:
                warnings.warn("visualisation trajectories are not produced for sharded controllers")
                self._viz_warned = True
        return u[0], u, optimal_traj, sampled

    def run_closed_loop(self, x0, n_ticks):
        """Closed loop on the device: tick, plant step (the reference's own plant for this controller), repeat.
        Equivalent to the reference's `for i in range(n): u0,... = ctrl._calc_...(x); x = plant(x, u0)` loops
        (mppi_differential_drive.py:305-367) without a host round trip per tick.  Needs waypoint_mode='frozen'."""
        plant = 1 if self.dim_x == 4 else 0
        states, controls = self._engine.run_closed_loop(np.asarray(x0, dtype=np.float64), int(n_ticks), self.seed,
                                                        self._tick, plant)
        self._tick += int(n_ticks)
        self._u_cache = self._engine.get_nominal().astype(self._out_dtype)
        return states.astype(self._out_dtype), controls.astype(self._out_dtype)

    def _viz_gates(self):
        """(replay the nominal?, replay the samples?) -- the diff-drive class gates both on visualze_sampled_trajs
        (mppi_differential_drive.py:145,154), the race-car class uses one flag each (:112,:121)."""
        return bool(self.visualze_sampled_trajs), bool(self.visualze_sampled_trajs)

    def comm_init_from_torch(self, exchange="p2p"):
        """Sample sharding over the torch.distributed ranks of one node.  exchange='p2p' (default): the
        (min, sum w, sum w*eps) exchange is fused into the tick kernel over NVLink peer memory (CUDA IPC
        handles all-gathered here); exchange='nccl': tick kernel, ncclAllGather, merge kernel."""
        import torch.distributed as dist
        rank, world = dist.get_rank(), dist.get_world_size()
        if exchange == "p2p":
            mine = self._engine.comm_p2p_export(world)
            handles = [None] * world
            dist.all_gather_object(handles, mine)
            self._engine.comm_p2p_open(b"".join(handles), rank, world)
            dist.barrier()
        elif exchange == "nccl":
            ids = [MPPIEngine.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(ids, src=0)
            self._engine.comm_init(ids[0], rank, world)
        else:
            raise ValueError("exchange must be 'p2p' or 'nccl'")

    @property
    def engine(self):
        return self._engine
