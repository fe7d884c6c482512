"""Thin host-side wrapper of one libmppi_b200 handle.  PyTorch is used only for device
memory of user-supplied tensors (injected noise, batched states); all compute is in the
hand-written sm_100a kernels behind the C ABI."""
import ctypes as C
import math

import numpy as np

from . import _lib


def _dptr(t):
    """Device pointer of a torch CUDA tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


class MPPIEngine:
    """One controller (or a batch of R controllers) bound to one GPU."""

    def __init__(self, *, model, K, T, dt, u_max, sigma, stage_w, term_w, param_exploration,
                 param_lambda, param_alpha, temperature, window, cost_mode, waypoint_mode,
                 filter_kind, yaw_wrap, collision="none", obstacles=None, margin=1.0,
                 wheel_base=2.5, robot_radius=0.5, vehicle_l=4.0, vehicle_w=3.0, n_robots=1,
                 device=0, K_global=None, k_offset=0, clamp_nominal=False, cost_kind="path", goal=None,
                 ctrl_w=None, soft_obs_weight=None, soft_obs_safety=None):
        self.lib = _lib.load()
        c = _lib.MppiConfig()
        self.lib.mppi_default_config(C.byref(c))
        c.device = int(device)
        c.model = _lib.MODEL[model]
        c.K, c.T, c.n_robots, c.window = int(K), int(T), int(n_robots), int(window)
        c.cost_mode = _lib.COST_MODE[cost_mode]
        c.waypoint_mode = _lib.WAYPOINT_MODE[waypoint_mode]
        c.filter_kind = _lib.FILTER[filter_kind]
        c.yaw_wrap = int(bool(yaw_wrap))
        c.collision = _lib.COLLISION[collision]
        c.K_global = int(K_global) if K_global else int(K)
        c.k_offset = int(k_offset)
        c.clamp_nominal = int(bool(clamp_nominal))
        c.cost_kind = _lib.COST_KIND[cost_kind]
        if goal is not None:
            g = np.zeros(4); g[:len(goal)] = np.asarray(goal, float)
            c.goal[:] = list(g)
        if ctrl_w is not None:
            c.ctrl_w[:] = [float(ctrl_w[0]), float(ctrl_w[1])]
        if soft_obs_weight is not None:
            c.soft_obs_weight = float(soft_obs_weight)
        if soft_obs_safety is not None:
            c.soft_obs_safety = float(soft_obs_safety)
        c.dt, c.wheel_base = float(dt), float(wheel_base)
        c.u_max[:] = [float(u_max[0]), float(u_max[1])]
        c.param_exploration, c.param_lambda, c.param_alpha = float(param_exploration), float(param_lambda), float(param_alpha)
        c.temperature = float(temperature)
        c.sigma[:] = [float(v) for v in np.asarray(sigma, float).reshape(4)]
        sw = np.zeros(4); sw[:len(stage_w)] = np.asarray(stage_w, float)
        tw = np.zeros(4); tw[:len(term_w)] = np.asarray(term_w, float)
        c.stage_w[:] = list(sw)
        c.term_w[:] = list(tw)
        c.margin, c.robot_radius, c.vehicle_l, c.vehicle_w = float(margin), float(robot_radius), float(vehicle_l), float(vehicle_w)
        self.cfg = c
        self.K, self.T, self.R = int(K), int(T), int(n_robots)
        self.nx = 4 if model == "bicycle" else 3
        self.model = model
        self.device = int(device)
        self._h = C.c_void_p()
        st = self.lib.mppi_create(C.byref(c), C.byref(self._h))
        if st != 0:
            self._h = C.c_void_p()
            raise _lib.MppiError("mppi_create failed: %s (no CUDA device, or invalid configuration; "
                                 "this engine has no CPU fallback)" % self.lib.mppi_strerror(st).decode())
        # preallocated host staging: one ctypes call per tick, no per-call allocation
        self._x0 = (C.c_double * 4)()
        self._u0 = (C.c_float * 2)()
        self._useq = (C.c_float * (2 * self.T))()
        self._useq_np = np.frombuffer(self._useq, dtype=np.float32).reshape(self.T, 2)
        self._u0_np = np.frombuffer(self._u0, dtype=np.float32)
        # the shared scene as last set (use_shared_scene re-installs it after per-robot goals / obstacles)
        self._cost_kind, self._collision = cost_kind, collision
        self._shared_goal = np.asarray(c.goal[:2 if cost_kind == "goal" else 3], dtype=np.float64)
        self._shared_obs = np.zeros((0, 3))
        self._shared_moving = (np.zeros((0, 2)), np.zeros((0, 2)))
        if obstacles is not None and len(obstacles):
            self.set_obstacles(obstacles)

    # -- lifecycle -------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.mppi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, st, what):
        _lib.check(self.lib, self._h, st, what)

    # -- state -----------------------------------------------------------------------------
    def set_ref_path(self, path):
        p = np.ascontiguousarray(path, dtype=np.float64)
        self._ck(self.lib.mppi_set_ref_path(self._h, p.ctypes.data_as(_lib._PD), p.shape[0], p.shape[1]), "mppi_set_ref_path")

    def set_ref_paths_spline(self, d_wx, d_wy, ds=0.1, max_points=512):
        """Per-robot courses generated on the device from (R, n_wp) float32 CUDA waypoint tensors (the reference's
        calc_spline_course, path_generator/cubic_spline_planner.py:311-323)."""
        if tuple(d_wx.shape) != tuple(d_wy.shape) or d_wx.shape[0] != self.R or not (d_wx.is_contiguous() and d_wy.is_contiguous()):
            raise ValueError("waypoints must be contiguous (R, n_wp) float32 CUDA tensors")
        self._ck(self.lib.mppi_set_ref_paths_spline(self._h, _dptr(d_wx), _dptr(d_wy), int(d_wx.shape[1]), float(ds),
                                                    int(max_points)), "mppi_set_ref_paths_spline")

    def get_ref_path(self, robot=0):
        n = C.c_int32(0)
        self._ck(self.lib.mppi_get_ref_path(self._h, int(robot), None, 0, C.byref(n)), "mppi_get_ref_path")
        out = np.zeros((n.value, 4), dtype=np.float32)
        self._ck(self.lib.mppi_get_ref_path(self._h, int(robot), out.ctypes.data_as(_lib._PF), n.value, C.byref(n)),
                 "mppi_get_ref_path")
        return out

    def set_obstacles(self, obstacles):
        o = np.ascontiguousarray(obstacles, dtype=np.float64).reshape(-1, 3)
        self._ck(self.lib.mppi_set_obstacles(self._h, o.ctypes.data_as(_lib._PD), o.shape[0]), "mppi_set_obstacles")
        self._shared_obs = o.copy()

    def set_goal(self, goal):
        g = np.ascontiguousarray(goal, dtype=np.float64).reshape(-1)
        self._ck(self.lib.mppi_set_goal(self._h, g.ctypes.data_as(_lib._PD), g.shape[0]), "mppi_set_goal")
        self._shared_goal = g.copy()

    def set_moving_obstacles(self, pos_xy, vel_xy):
        p = np.ascontiguousarray(pos_xy, dtype=np.float64).reshape(-1, 2)
        v = np.ascontiguousarray(vel_xy, dtype=np.float64).reshape(-1, 2)
        if p.shape != v.shape:
            raise ValueError("positions and velocities must both be (M,2)")
        self._ck(self.lib.mppi_set_moving_obstacles(self._h, p.ctypes.data_as(_lib._PD), v.ctypes.data_as(_lib._PD), p.shape[0]),
                 "mppi_set_moving_obstacles")
        self._shared_moving = (p.copy(), v.copy())

    def use_shared_scene(self):
        """Drops per-robot goals / obstacles: every robot scores against the shared goal and obstacle set last given to the
        constructor or to set_goal / set_obstacles / set_moving_obstacles."""
        if self._cost_kind != "path":
            self.set_goal(self._shared_goal)
        if self._cost_kind == "target_soft":
            self.set_moving_obstacles(*self._shared_moving)
        elif self._collision != "none":
            self.set_obstacles(self._shared_obs)

    def _device_rows(self, a, dtype, shape, what):
        """(tensor, uploaded) for a per-robot argument: a CUDA tensor is used as it is (read by a kernel on the engine's
        stream), a host array is uploaded and the upload is waited for."""
        import torch
        if isinstance(a, torch.Tensor) and a.is_cuda:
            if a.dtype != dtype or not a.is_contiguous() or tuple(a.shape) != shape or a.device.index != self.device:
                raise ValueError("%s must be a contiguous %s CUDA tensor of shape %s on cuda:%d" % (what, dtype, shape, self.device))
            return a, False
        t = torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda:%d" % self.device).contiguous()
        if tuple(t.shape) != shape:
            raise ValueError("%s must have shape %s" % (what, shape))
        torch.cuda.current_stream(self.device).synchronize()      # the upload is complete before the engine's stream reads it
        return t, True

    def _after_upload(self, uploaded):
        if uploaded:                                             # the staged copy must outlive the install kernel
            import torch
            torch.cuda.synchronize(self.device)

    def set_robot_obstacles(self, obs, counts=None):
        """One obstacle set PER ROBOT: obs (R, m, 3) static circles [x, y, r] (circle / footprint collision) or (R, m, 4)
        moving soft obstacles [x, y, vx, vy] (target_soft), m <= 16; counts (R,) int32: robot r uses its first counts[r]
        rows (default: all m).  A CUDA tensor is read by a kernel enqueued on the engine's stream, without a host
        synchronisation: whatever writes it must be ordered before that stream's work (BatchedMPPI runs the engine on torch's
        current stream, so torch work issued before the call is; a bare engine runs on its own stream unless set_stream
        is called).  A numpy array is uploaded, which synchronises the device."""
        import torch
        shape = tuple(obs.shape)
        if len(shape) != 3 or shape[0] != self.R or shape[2] not in (3, 4):
            raise ValueError("obstacles must be (R, m, 3) or (R, m, 4)")
        d_obs, up1 = self._device_rows(obs, torch.float32, shape, "obstacles")
        d_cnt, up2 = (None, False) if counts is None else self._device_rows(counts, torch.int32, (self.R,), "counts")
        self._ck(self.lib.mppi_set_robot_obstacles(self._h, _dptr(d_obs), _dptr(d_cnt), shape[1], shape[2]),
                 "mppi_set_robot_obstacles")
        self._after_upload(up1 or up2)

    def set_robot_goals(self, goals):
        """One goal PER ROBOT: (R, 2) goal points (goal cost kind) or (R, 3) target poses (target_soft).  CUDA tensors and
        numpy arrays are consumed as by set_robot_obstacles."""
        import torch
        shape = tuple(goals.shape)
        if len(shape) != 2 or shape[0] != self.R:
            raise ValueError("goals must be (R, 2) or (R, 3)")
        d_goal, up = self._device_rows(goals, torch.float32, shape, "goals")
        self._ck(self.lib.mppi_set_robot_goals(self._h, _dptr(d_goal), shape[1]), "mppi_set_robot_goals")
        self._after_upload(up)

    def set_nominal(self, u):
        u = np.ascontiguousarray(u, dtype=np.float32).reshape(self.R * self.T * 2)
        self._ck(self.lib.mppi_set_nominal(self._h, u.ctypes.data_as(_lib._PF)), "mppi_set_nominal")

    def get_nominal(self):
        u = np.zeros(self.R * self.T * 2, dtype=np.float32)
        self._ck(self.lib.mppi_get_nominal(self._h, u.ctypes.data_as(_lib._PF)), "mppi_get_nominal")
        return u.reshape(self.T, 2) if self.R == 1 else u.reshape(self.R, self.T, 2)

    def set_waypoint_idx(self, idx):
        a = np.ascontiguousarray(np.broadcast_to(np.asarray(idx, dtype=np.int32), (self.R,)))
        self._ck(self.lib.mppi_set_waypoint_idx(self._h, a.ctypes.data_as(_lib._PI)), "mppi_set_waypoint_idx")

    def get_waypoint_idx(self):
        a = np.zeros(self.R, dtype=np.int32)
        self._ck(self.lib.mppi_get_waypoint_idx(self._h, a.ctypes.data_as(_lib._PI)), "mppi_get_waypoint_idx")
        return int(a[0]) if self.R == 1 else a

    def set_mlp(self, weights, biases, in_mean=None, in_scale=None, out_mean=None, out_scale=None):
        """nn.Linear-layout weights of the residual MLP: input layer (512, n_in) with n_in = 3 (state, dnn/simple_mlp.py)
        or 5 (state + control, the trained saved_models), hidden layers (512, 512), output layer (3, 512); optional
        StandardScaler statistics folded into the first / last layer."""
        Ws = [np.ascontiguousarray(w, dtype=np.float32) for w in weights]
        bs = [np.ascontiguousarray(b, dtype=np.float32) for b in biases]
        n = len(Ws)
        Wp = (_lib._PF * n)(*[w.ctypes.data_as(_lib._PF) for w in Ws])
        bp = (_lib._PF * n)(*[b.ctypes.data_as(_lib._PF) for b in bs])
        n_in = int(Ws[0].shape[1])
        if n == 4 and n_in == 3 and in_mean is None and in_scale is None and out_mean is None and out_scale is None:
            self._ck(self.lib.mppi_set_mlp(self._h, Wp, bp), "mppi_set_mlp")
            return

        def vec(v, k):
            if v is None:
                return None, None
            a = np.ascontiguousarray(v, dtype=np.float64).reshape(k)
            return a, a.ctypes.data_as(_lib._PD)
        keep = [vec(in_mean, n_in), vec(in_scale, n_in), vec(out_mean, 3), vec(out_scale, 3)]
        self._ck(self.lib.mppi_set_mlp_ex(self._h, n_in, n - 2, Wp, bp, *[k[1] for k in keep]), "mppi_set_mlp_ex")

    # -- ticks -----------------------------------------------------------------------------
    def _load_x0(self, x0):
        for i in range(self.nx):
            self._x0[i] = float(x0[i])

    def step(self, x0, d_eps=None, seed=0, tick=0):
        """One control tick; returns views (u0 (2,), u_seq (T,2)) of internal float32 staging."""
        self._load_x0(x0)
        st = self.lib.mppi_step(self._h, self._x0, _dptr(d_eps), seed, tick, self._u0, self._useq)
        if st != 0:
            self._ck(st, "mppi_step")
        return self._u0_np, self._useq_np

    def step_async(self, x0, d_eps=None, seed=0, tick=0):
        self._load_x0(x0)
        self._ck(self.lib.mppi_step_async(self._h, self._x0, _dptr(d_eps), seed, tick), "mppi_step_async")

    def synchronize(self):
        self._ck(self.lib.mppi_synchronize(self._h), "mppi_synchronize")

    def rollout_costs(self, x0, d_S, d_eps=None, seed=0, tick=0):
        self._load_x0(x0)
        self._ck(self.lib.mppi_rollout_costs(self._h, self._x0, _dptr(d_eps), seed, tick, _dptr(d_S)), "mppi_rollout_costs")

    def reduce_update(self, d_S, d_eps=None, seed=0, tick=0):
        w_eps = np.zeros((self.T, 2), dtype=np.float32)
        self._ck(self.lib.mppi_reduce_update(self._h, _dptr(d_S), _dptr(d_eps), seed, tick, self._u0, self._useq,
                                             w_eps.ctypes.data_as(_lib._PF)), "mppi_reduce_update")
        return self._u0_np.copy(), self._useq_np.copy(), w_eps

    def trajectories(self, x0, d_sampled=None, want_optimal=True, d_eps=None, seed=0, tick=0):
        """Visualisation replays of the tick just stepped (same x0 / noise source).  Returns the (T,nx) optimal
        trajectory (float32) or None; `d_sampled` (K,T,nx) CUDA tensor is filled when given."""
        self._load_x0(x0)
        opt = np.zeros((self.T, self.nx), dtype=np.float32) if want_optimal else None
        self._ck(self.lib.mppi_get_trajectories(self._h, self._x0, _dptr(d_eps), seed, tick,
                                                opt.ctypes.data_as(_lib._PF) if want_optimal else None, _dptr(d_sampled)),
                 "mppi_get_trajectories")
        return opt

    def set_keep_costs(self, on=True):
        self._ck(self.lib.mppi_set_keep_costs(self._h, int(on)), "mppi_set_keep_costs")

    def top_trajectories(self, x0, d_traj, n_top, d_idx=None, d_cost=None, want_optimal=False, index_shift=1,
                         d_eps=None, seed=0, tick=0):
        """The n_top lowest-cost samples of the tick just stepped, replayed into `d_traj` (n_top,T,nx) in ascending cost
        order; needs set_keep_costs(True) before the step.  Returns the (T,nx) optimal replay or None."""
        self._load_x0(x0)
        opt = np.zeros((self.T, self.nx), dtype=np.float32) if want_optimal else None
        self._ck(self.lib.mppi_get_top_trajectories(self._h, self._x0, _dptr(d_eps), seed, tick, int(n_top), int(index_shift),
                                                    opt.ctypes.data_as(_lib._PF) if want_optimal else None,
                                                    _dptr(d_traj), _dptr(d_idx), _dptr(d_cost)), "mppi_get_top_trajectories")
        return opt

    def generate_noise(self, d_out, seed=0, tick=0, robot=0):
        self._ck(self.lib.mppi_generate_noise_robot(self._h, seed, tick, robot, _dptr(d_out)), "mppi_generate_noise")

    def run_closed_loop(self, x0, n_ticks, seed=0, tick0=0, plant=0):
        """n_ticks control ticks with the plant step on the device between them (one CUDA graph).  Returns (states
        (n+1,nx), controls (n,2)) float32; for a fleet handle (n_robots = R, x0 (R,nx)): (n+1,R,nx) and (n,R,2)."""
        x = np.ascontiguousarray(np.asarray(x0, dtype=np.float64).reshape(self.R, -1)[:, :self.nx])
        states = np.zeros((n_ticks + 1, self.R, self.nx), dtype=np.float32)
        controls = np.zeros((n_ticks, self.R, 2), dtype=np.float32)
        self._ck(self.lib.mppi_run_closed_loop(self._h, x.ctypes.data_as(_lib._PD), n_ticks, seed, tick0, plant,
                                               states.ctypes.data_as(_lib._PF), controls.ctypes.data_as(_lib._PF)),
                 "mppi_run_closed_loop")
        if self.R == 1:
            return states[:, 0], controls[:, 0]
        return states, controls

    def step_batched(self, d_x0, d_u0_out=None, seed=0, tick=0):
        self._ck(self.lib.mppi_step_batched(self._h, _dptr(d_x0), seed, tick, _dptr(d_u0_out)), "mppi_step_batched")

    def stats(self):
        s = _lib.MppiStats()
        self._ck(self.lib.mppi_get_stats(self._h, C.byref(s)), "mppi_get_stats")
        return dict(rho=s.rho, eta=s.eta, ess=s.ess, min_collisions=s.min_collisions, idx=s.idx,
                    u_first=np.array([s.u_first[0], s.u_first[1]], dtype=np.float32))

    def set_trace(self, on=True):
        self._ck(self.lib.mppi_set_trace(self._h, int(on)), "mppi_set_trace")

    def trace(self):
        """Per-CTA (start, rollouts-done) %globaltimer stamps of the last tick and the last CTA's (merged, updated) pair."""
        buf = (C.c_uint64 * 4096)()
        n = C.c_int32(0)
        self._ck(self.lib.mppi_get_trace(self._h, buf, 4096, C.byref(n)), "mppi_get_trace")
        a = np.frombuffer(buf, dtype=np.uint64)[:2 * (n.value + 1)].astype(np.int64).reshape(-1, 2)
        return a[:n.value], a[n.value]

    def check_guards(self):
        """Number of device buffers whose guard zone was overwritten (0 = clean)."""
        n = self.lib.mppi_debug_check_guards(self._h)
        if n < 0:
            self._ck(n, "mppi_debug_check_guards")
        return n

    def set_timing(self, on=True):
        self._ck(self.lib.mppi_set_timing(self._h, int(on)), "mppi_set_timing")

    def timings(self):
        t = _lib.MppiTimings()
        self._ck(self.lib.mppi_get_timings(self._h, C.byref(t)), "mppi_get_timings")
        return dict(last_step_ms=t.last_step_ms, last_rollout_ms=t.last_rollout_ms,
                    last_update_ms=t.last_update_ms, last_passes=t.last_passes, launches=t.launches)

    def set_stream(self, cuda_stream_ptr):
        self._ck(self.lib.mppi_set_stream(self._h, C.c_void_p(cuda_stream_ptr)), "mppi_set_stream")

    # -- sample sharding -------------------------------------------------------------------
    def comm_init(self, unique_id: bytes, rank: int, world: int):
        buf = C.create_string_buffer(unique_id, 128)
        self._ck(self.lib.mppi_comm_init(self._h, buf, rank, world), "mppi_comm_init")

    def comm_p2p_export(self, world: int) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(self.lib.mppi_comm_p2p_export(self._h, world, buf), "mppi_comm_p2p_export")
        return buf.raw

    def comm_p2p_open(self, handles: bytes, rank: int, world: int):
        buf = C.create_string_buffer(handles, 64 * world)
        self._ck(self.lib.mppi_comm_p2p_open(self._h, buf, rank, world), "mppi_comm_p2p_open")

    def comm_p2p_barrier(self):
        """Device-side barrier of the sharding ranks, enqueued on the engine's stream (asynchronous)."""
        self._ck(self.lib.mppi_comm_p2p_barrier(self._h), "mppi_comm_p2p_barrier")

    def comm_p2p_trace(self):
        """%globaltimer stamps (ns) of the last fused exchange: local merge done, words stored, all ranks seen, updated."""
        t = (C.c_uint64 * 4)()
        self._ck(self.lib.mppi_comm_p2p_trace(self._h, t), "mppi_comm_p2p_trace")
        return [int(v) for v in t]

    @staticmethod
    def comm_unique_id() -> bytes:
        lib = _lib.load()
        buf = C.create_string_buffer(128)
        st = lib.mppi_comm_get_unique_id(buf)
        if st != 0:
            raise _lib.MppiError("mppi_comm_get_unique_id failed: %s" % lib.mppi_strerror(st).decode())
        return buf.raw


def n_exploit(param_exploration, K):
    """Q6: #{k : k < (1.0 - param_exploration) * K} evaluated like the reference (Python floats)."""
    return max(0, min(K, int(math.ceil((1.0 - param_exploration) * K))))
