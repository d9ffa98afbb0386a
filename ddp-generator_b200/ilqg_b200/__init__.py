"""Host-side Python mirror of the C ABI in include/ilqg_b200.h (ctypes; no torch types in any signature).

Usage mirrors the reference's mex call `[success, x, u, cost] = iLQG<Name>(x0, u0, p, Op)` (iLQG_mex.c:19-33) for a
whole batch:

    s = BatchSolver("car", full_ddp=0, batch=B, n_hor=T)
    s.set_options({"max_iter": 50}); s.set_params(params)
    out = s.solve(x0, u0)        # dict: success, x, u, cost, iterations, n_linesearch

The shared library is the product; if it is missing or no GPU is usable, construction raises -- there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_DIR = os.environ.get("ILQG_LIB_DIR") or os.path.join(os.path.dirname(_HERE), "lib")
TRACE, TIMING = 1, 2
KERNEL_CLASSES = ("derivs", "backpass", "linesearch", "post")
_SCALAR_FIELDS = {"cost", "new_cost", "dcost", "expected", "lambda", "dlambda", "g_norm", "dV0", "dV1", "w_pen_l", "w_pen_f",
                  "iterations", "result", "status", "n_linesearch", "n_backpass", "n_derivs", "n_rollouts", "n_tails", "cur", "bp_split",
                  "cw_lpp", "bp_latency", "ls_tail_from", "ls_commit_par", "policy_ok"}


def lib_path(problem, full_ddp, lib_dir=None):
    return os.path.join(lib_dir or LIB_DIR, f"libilqg_b200_{problem}_ddp{int(full_ddp)}.so")


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Library:
    """One loaded libilqg_b200_<problem>_ddp<d>.so with typed entry points."""

    _cache = {}

    def __new__(cls, problem, full_ddp, lib_dir=None):
        key = (problem, int(full_ddp), lib_dir)
        if key not in cls._cache:
            self = super().__new__(cls)
            self._load(problem, full_ddp, lib_dir)
            cls._cache[key] = self
        return cls._cache[key]

    def _load(self, problem, full_ddp, lib_dir=None):
        path = lib_path(problem, full_ddp, lib_dir)
        if not os.path.exists(path):
            raise RuntimeError(f"{path} not found: build it with `make -C ddp-generator_b200` (no CPU fallback exists)")
        L = self.lib = C.CDLL(path)
        self.path = path
        vp, cp, ci, dp = C.c_void_p, C.c_char_p, C.c_int, C.c_void_p
        L.ilqgb_problem_name.restype = cp
        L.ilqgb_param_name.restype = cp
        L.ilqgb_param_name.argtypes = [ci]
        L.ilqgb_param_size.argtypes = [ci]
        L.ilqgb_create.restype = vp
        L.ilqgb_create.argtypes = [ci, ci, ci, ci, vp]
        L.ilqgb_create_multi.restype = vp
        L.ilqgb_create_multi.argtypes = [ci, vp, ci, ci, ci, vp]
        L.ilqgb_devices.argtypes = [vp]
        L.ilqgb_destroy.argtypes = [vp]
        L.ilqgb_last_error.restype = cp
        L.ilqgb_last_error.argtypes = [vp]
        L.ilqgb_standard_parameters.argtypes = [vp]
        L.ilqgb_set_opt.restype = cp
        L.ilqgb_set_opt.argtypes = [vp, cp, dp, ci]
        L.ilqgb_set_param.argtypes = [vp, ci, dp, ci]
        L.ilqgb_set_param_batch.argtypes = [vp, ci, dp, ci]
        L.ilqgb_set_param_track.argtypes = [vp, ci, dp, ci]
        L.ilqgb_set_plant_param.argtypes = [vp, ci, dp, ci]
        L.ilqgb_set_plant_param_batch.argtypes = [vp, ci, dp, ci]
        L.ilqgb_set_plant_substeps.argtypes = [vp, ci]
        L.ilqgb_clear_plant.argtypes = [vp]
        L.ilqgb_set_track_offset.argtypes = [vp, ci]
        L.ilqgb_track_offset.argtypes = [vp]
        L.ilqgb_validate_opt.restype = cp
        L.ilqgb_validate_opt.argtypes = [cp, dp, ci]
        L.ilqgb_upload.argtypes = [vp, dp, dp]
        for f in ("ilqgb_start", "ilqgb_finish", "ilqgb_solve", "ilqgb_sync", "ilqgb_active", "ilqgb_phase_derivs",
                  "ilqgb_phase_backpass", "ilqgb_phase_linesearch"):
            getattr(L, f).argtypes = [vp]
        L.ilqgb_iterate.argtypes = [vp, ci]
        L.ilqgb_download.argtypes = [vp, dp, dp, dp, dp, dp, dp]
        L.ilqgb_solve_host.argtypes = [vp, dp, dp, dp, dp, dp, dp, dp, dp]
        L.ilqgb_shift.argtypes = [vp, ci, dp, dp]
        L.ilqgb_mpc.argtypes = [vp, ci, dp, dp, dp, dp, dp, dp, dp, dp]
        L.ilqgb_get.restype = C.c_long
        L.ilqgb_get.argtypes = [vp, cp, dp]
        L.ilqgb_get_int.restype = C.c_long
        L.ilqgb_get_int.argtypes = [vp, cp, dp]
        L.ilqgb_timing.argtypes = [vp, dp, dp, ci]
        L.ilqgb_launch_count.restype = C.c_long
        L.ilqgb_launch_count.argtypes = [vp]
        L.ilqgb_chunks.argtypes = [vp]
        L.ilqgb_set_tuning.argtypes = [vp, cp, ci]
        L.ilqgb_policy.argtypes = [vp]
        L.ilqgb_policy_rollout.argtypes = [vp, ci, dp, dp, dp, dp, dp, dp]
        L.ilqgb_policy_eval.argtypes = [vp, ci, dp, dp]
        self.problem = L.ilqgb_problem_name().decode()
        self.nx, self.nu = L.ilqgb_nx(), L.ilqgb_nu()
        self.full_ddp = L.ilqgb_full_ddp()
        self.param_names = [L.ilqgb_param_name(i).decode() for i in range(L.ilqgb_n_params())]
        self.param_sizes = [L.ilqgb_param_size(i) for i in range(L.ilqgb_n_params())]
        self.deriv_doubles_per_step = L.ilqgb_deriv_doubles_per_step()

    def validate_option(self, name, value):
        """setOptParam's check without a handle: None or the reference's message."""
        v = np.ascontiguousarray(np.atleast_1d(np.asarray(value, dtype=np.float64)))
        err = self.lib.ilqgb_validate_opt(name.encode(), _ptr(v), v.size)
        return err.decode() if err else None

    def device_count(self):
        return self.lib.ilqgb_device_count()


class BatchSolver:
    def __init__(self, problem, full_ddp=0, batch=1, n_hor=1, device=0, flags=0, stream=None, chunks=0, devices=None, lib_dir=None):
        """`devices`: list of GPU indices (or a count) to shard the batch over in this one process (ilqgb_create_multi);
        `chunks` then counts chunks per device.  Default: the single GPU `device`.  `lib_dir`: where the problem's library was
        built (python -m ilqg_gen.make --out DIR puts it in DIR/lib); default: the package's lib/."""
        self.L = Library(problem, full_ddp, lib_dir)
        self.lib = self.L.lib
        self.B, self.T = int(batch), int(n_hor)
        self.nx, self.nu = self.L.nx, self.L.nu
        self.max_iter = 20
        fl = int(flags) | ((int(chunks) & 0xff) << 8)
        st = C.c_void_p(stream) if stream else None
        if devices is None:
            self.h = self.lib.ilqgb_create(int(device), self.B, self.T, fl, st)
        else:
            devs = list(range(devices)) if isinstance(devices, int) else [int(d) for d in devices]
            arr = (C.c_int * len(devs))(*devs)
            self.h = self.lib.ilqgb_create_multi(len(devs), arr, self.B, self.T, fl, st)
        if not self.h:
            raise RuntimeError("ilqgb_create failed: " + self.lib.ilqgb_last_error(None).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.ilqgb_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def _chk(self, rc):
        if rc < 0:
            raise RuntimeError(self.lib.ilqgb_last_error(self.h).decode())
        return rc

    # options / parameters ------------------------------------------------------------------------------------------
    def set_option(self, name, value):
        """Returns None or the reference's error message (setOptParam semantics)."""
        v = np.ascontiguousarray(np.atleast_1d(np.asarray(value, dtype=np.float64)))
        err = self.lib.ilqgb_set_opt(self.h, name.encode(), _ptr(v), v.size)
        if err is None and name == "max_iter":
            self.max_iter = int(v[0])
        return err.decode() if err else None

    def set_options(self, opts):
        for k, v in opts.items():
            err = self.set_option(k, v)
            if err:
                raise ValueError(f"Error setting optimization parameter '{k}': {err}.")

    def set_params(self, params):
        for i, name in enumerate(self.L.param_names):
            if name not in params:
                raise KeyError(f"Parameter name '{name}' is not member of parameters struct.")
            v = np.ascontiguousarray(np.asarray(params[name], dtype=np.float64).ravel())
            self._chk(self.lib.ilqgb_set_param(self.h, i, _ptr(v), v.size))

    def set_params_batch(self, params):
        """Per-problem parameter sets: {name: array [batch, size]} for the names that differ between problems."""
        for name, val in params.items():
            i = self.L.param_names.index(name)
            v = np.ascontiguousarray(np.asarray(val, dtype=np.float64).reshape(self.B, -1))
            self._chk(self.lib.ilqgb_set_param_batch(self.h, i, _ptr(v), v.shape[1]))

    def set_param_track(self, name, values):
        """A track per problem for the [k]-indexed parameter `name`: values [batch, len], len >= n_hor + 1 (ilqgb_set_param_track).
        A solve reads name[k] = values[b, offset + k]; shift() and mpc() move the offset with the plan.  set_params() with
        this name makes the parameter shared again."""
        i = self.L.param_names.index(name)
        v = np.ascontiguousarray(np.asarray(values, dtype=np.float64))
        if v.ndim != 2 or v.shape[0] != self.B:
            raise ValueError(f"track of '{name}' must be [batch, len] = [{self.B}, >= {self.T + 1}], got {list(v.shape)}")
        self._chk(self.lib.ilqgb_set_param_track(self.h, i, _ptr(v), v.shape[1]))

    def set_track_offset(self, n):
        """Window offset of every track: the next solve reads values[b, n + k] (ilqgb_set_track_offset)."""
        self._chk(self.lib.ilqgb_set_track_offset(self.h, int(n)))

    def track_offset(self):
        return int(self.lib.ilqgb_track_offset(self.h))

    # plant of the closed loops -------------------------------------------------------------------------------------------
    def _param_index(self, name):
        if name not in self.L.param_names:
            raise KeyError(f"Parameter name '{name}' is not member of parameters struct.")
        return self.L.param_names.index(name)

    def set_plant_params(self, params):
        """The plant's own shared values {name: value} (ilqgb_set_plant_param); names not given follow the model.  With a plant,
        shift() and mpc() step the next x0 from the solve's x0 through the applied controls with these parameters instead of
        taking the solution's prediction.  [k]-indexed parameters are always the model's."""
        for name, val in params.items():
            v = np.ascontiguousarray(np.asarray(val, dtype=np.float64).ravel())
            self._chk(self.lib.ilqgb_set_plant_param(self.h, self._param_index(name), _ptr(v), v.size))

    def set_plant_params_batch(self, params):
        """Per-problem plant values {name: array [batch, size]} (ilqgb_set_plant_param_batch)."""
        for name, val in params.items():
            i = self._param_index(name)
            size = self.L.param_sizes[i]
            v = np.ascontiguousarray(np.asarray(val, dtype=np.float64))
            if v.ndim == 1 and size == 1:
                v = v[:, None]
            if v.shape != (self.B, size):
                raise ValueError(f"plant values of '{name}' must be [batch, size] = [{self.B}, {size}], got {list(v.shape)}")
            self._chk(self.lib.ilqgb_set_plant_param_batch(self.h, i, _ptr(v), size))

    def set_plant_substeps(self, n_sub):
        """Plant steps per control interval, 1..64.  Nothing is rescaled: set the plant's time step to the model's / n_sub."""
        self._chk(self.lib.ilqgb_set_plant_substeps(self.h, int(n_sub)))

    def clear_plant(self):
        """No plant: the next x0 is the solution's prediction x[n] (+ w) again."""
        self._chk(self.lib.ilqgb_clear_plant(self.h))

    # data ----------------------------------------------------------------------------------------------------------------
    def upload(self, x0, u0):
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        u0 = np.ascontiguousarray(u0, dtype=np.float64)
        if x0.shape != (self.B, self.nx):
            raise ValueError(f"wrong number of elements in x0 ({self.B}x{self.nx} expected)")
        if u0.shape != (self.B, self.T, self.nu):
            raise ValueError(f"wrong number of elements in u_nom ({self.B}x{self.T}x{self.nu} expected)")
        self._chk(self.lib.ilqgb_upload(self.h, _ptr(x0), _ptr(u0)))
        self._keep = (x0, u0)

    def upload_ptr(self, x0_ptr, u0_ptr):
        self._chk(self.lib.ilqgb_upload(self.h, C.c_void_p(x0_ptr), C.c_void_p(u0_ptr)))

    def download(self, want_traj=True):
        x = np.empty((self.B, self.T + 1, self.nx)) if want_traj else None
        u = np.empty((self.B, self.T, self.nu)) if want_traj else None
        cost = np.empty(self.B)
        it = np.empty(self.B, np.int32)
        res = np.empty(self.B, np.int32)
        nls = np.empty(self.B, np.int32)
        self._chk(self.lib.ilqgb_download(self.h, _ptr(x), _ptr(u), _ptr(cost), _ptr(it), _ptr(res), _ptr(nls)))
        return dict(success=res, x=x, u=u, cost=cost, iterations=it, n_linesearch=nls)

    def download_ptr(self, x_ptr, u_ptr, cost_ptr, it_ptr, res_ptr, nls_ptr):
        self._chk(self.lib.ilqgb_download(self.h, *[C.c_void_p(p) if p else None for p in (x_ptr, u_ptr, cost_ptr, it_ptr, res_ptr, nls_ptr)]))

    # solve -------------------------------------------------------------------------------------------------------------
    def start(self):
        self._chk(self.lib.ilqgb_start(self.h))

    def iterate(self, n):
        return self._chk(self.lib.ilqgb_iterate(self.h, int(n)))

    def finish(self):
        self._chk(self.lib.ilqgb_finish(self.h))

    def run(self):
        self._chk(self.lib.ilqgb_solve(self.h))

    def sync(self):
        self._chk(self.lib.ilqgb_sync(self.h))

    def active(self):
        return self._chk(self.lib.ilqgb_active(self.h))

    def solve(self, x0, u0, want_traj=True):
        self.upload(x0, u0)
        self.run()
        return self.download(want_traj)

    def solve_host_ptr(self, x0_ptr, u0_ptr, x_ptr, u_ptr, cost_ptr, it_ptr, res_ptr, nls_ptr):
        """Pipelined upload + solve + download on raw host pointers (pinned memory for full overlap)."""
        self._chk(self.lib.ilqgb_solve_host(self.h, *[C.c_void_p(p) if p else None for p in (x0_ptr, u0_ptr, x_ptr, u_ptr, cost_ptr, it_ptr, res_ptr, nls_ptr)]))

    def solve_host(self, x0, u0):
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        u0 = np.ascontiguousarray(u0, dtype=np.float64)
        x = np.empty((self.B, self.T + 1, self.nx)); u = np.empty((self.B, self.T, self.nu)); cost = np.empty(self.B)
        it = np.empty(self.B, np.int32); res = np.empty(self.B, np.int32); nls = np.empty(self.B, np.int32)
        self._chk(self.lib.ilqgb_solve_host(self.h, _ptr(x0), _ptr(u0), _ptr(x), _ptr(u), _ptr(cost), _ptr(it), _ptr(res), _ptr(nls)))
        return dict(success=res, x=x, u=u, cost=cost, iterations=it, n_linesearch=nls)

    # receding horizon ----------------------------------------------------------------------------------------------------
    def _state(self, name, a, shape):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=np.float64)
        if a.shape != shape:
            raise ValueError(f"wrong number of elements in {name} ({'x'.join(map(str, shape))} expected)")
        return a

    def shift(self, n=1, x0=None, w=None):
        """The current solution becomes the next solve's input (ilqgb_shift): u[k] <- u[k+n], the last control repeated;
        x0 <- x0 if given, else x[n] (+ w [B, nx]).  Needs a start since the last upload or shift."""
        x0 = self._state("x0", x0, (self.B, self.nx))
        w = self._state("w", w, (self.B, self.nx))
        self._chk(self.lib.ilqgb_shift(self.h, int(n), _ptr(x0), _ptr(w)))
        self._keep = (x0, w)

    def mpc(self, x0, u0, n_steps, w=None):
        """n_steps closed-loop steps on the device (ilqgb_mpc): solve, apply u[0], x0 <- x[1] + w[:, step], shift by one.
        x0 = u0 = None continues from the current input (after upload or shift).  Returns the logs: x [B, S+1, nx] (the x0 of
        every solve, then the final state), u [B, S, nu] (applied controls), cost, iterations, success [B, S].  The handle then
        holds the last step's solution (download() returns the final plan)."""
        S = int(n_steps)
        if (x0 is None) != (u0 is None):
            raise ValueError("x0 and u0 go together (neither: continue from the current input)")
        x0 = self._state("x0", x0, (self.B, self.nx))
        u0 = self._state("u_nom", u0, (self.B, self.T, self.nu))
        w = self._state("w", w, (self.B, S, self.nx))
        out = dict(x=np.empty((self.B, S + 1, self.nx)), u=np.empty((self.B, S, self.nu)), cost=np.empty((self.B, S)),
                   iterations=np.empty((self.B, S), np.int32), success=np.empty((self.B, S), np.int32))
        self._chk(self.lib.ilqgb_mpc(self.h, S, _ptr(x0), _ptr(u0), _ptr(w), *[_ptr(out[k]) for k in ("x", "u", "cost", "iterations", "success")]))
        return out

    # feedback policy of a solved batch ------------------------------------------------------------------------------------
    def policy(self):
        """Gains at the final trajectory of every problem (ilqgb_policy): calc_derivs + one back_pass at the final lambda.
        get_int("policy_ok") says which problems got them.  Valid until the next upload, start, shift, mpc, solve or put."""
        self._chk(self.lib.ilqgb_policy(self.h))

    def policy_rollout(self, x0s, want_traj=False):
        """Closed-loop rollouts of the policy from x0s [B, M, nx] (ilqgb_policy_rollout): u = u*_k + L_k (x - x*_k), clamped, then
        the model's (or the plant's) dynamics.  Returns cost [B, M], x_final [B, M, nx], ok [B, M] and, with want_traj,
        x [B, M, T+1, nx] and u [B, M, T, nu].  The handle is left as it was."""
        x0s = np.ascontiguousarray(x0s, dtype=np.float64)
        if x0s.ndim != 3 or x0s.shape[0] != self.B or x0s.shape[2] != self.nx:
            raise ValueError(f"x0s must be [batch, M, nx] = [{self.B}, M, {self.nx}], got {list(x0s.shape)}")
        B, M = self.B, x0s.shape[1]
        out = dict(cost=np.empty((B, M)), x_final=np.empty((B, M, self.nx)), ok=np.empty((B, M), np.int32))
        if want_traj:
            out["x"] = np.empty((B, M, self.T + 1, self.nx))
            out["u"] = np.empty((B, M, self.T, self.nu))
        self._chk(self.lib.ilqgb_policy_rollout(self.h, M, _ptr(x0s), _ptr(out["cost"]), _ptr(out["x_final"]), _ptr(out["ok"]),
                                                _ptr(out.get("x")), _ptr(out.get("u"))))
        return out

    def policy_eval(self, k, x):
        """The policy's control at step k for one state per problem, x [B, nx] -> u [B, nu] (ilqgb_policy_eval)."""
        x = self._state("x", x, (self.B, self.nx))
        u = np.empty((self.B, self.nu))
        self._chk(self.lib.ilqgb_policy_eval(self.h, int(k), _ptr(x), _ptr(u)))
        return u

    def set_tuning(self, name, value):
        """Run-time tuning knobs (ilqgb_set_tuning): ls_tail_from, bp_latency, bp_split, cw_lpp, pass_index."""
        self._chk(self.lib.ilqgb_set_tuning(self.h, name.encode(), int(value)))

    def phase(self, which):
        self._chk(getattr(self.lib, f"ilqgb_phase_{which}")(self.h))

    # read-back ---------------------------------------------------------------------------------------------------------
    def get(self, field):
        """A per-problem field of ilqgb_get; "plant" is the effective plant parameter set [B, sum of parameter sizes]."""
        T, nx, nu, B = self.T, self.nx, self.nu, self.B
        nq = nx * (nx + 1) // 2
        shapes = {"x": (B, T + 1, nx), "u": (B, T, nu), "l": (B, T, nu), "L": (B, T, nu * nx), "fd": (B, nx + nq)}
        n_max = B * max((T + 1) * max(nx * nu, self.L.deriv_doubles_per_step, nx, 4), self.max_iter + 1) + 64
        buf = np.empty(n_max)
        n = self._chk(self.lib.ilqgb_get(self.h, field.encode(), _ptr(buf)))
        out = buf[:n].copy()
        if field in shapes:
            return out.reshape(shapes[field])
        return out if field in _SCALAR_FIELDS else out.reshape(B, -1)

    def get_int(self, field):
        n_max = self.B * max(self.T, self.max_iter + 1) + 64
        buf = np.empty(n_max, np.int32)
        n = self._chk(self.lib.ilqgb_get_int(self.h, field.encode(), _ptr(buf)))
        out = buf[:n].copy()
        return out if field in _SCALAR_FIELDS else out.reshape(self.B, -1)

    def chunks(self):
        return int(self.lib.ilqgb_chunks(self.h))

    def devices(self):
        return int(self.lib.ilqgb_devices(self.h))

    def launch_count(self):
        return int(self.lib.ilqgb_launch_count(self.h))

    def timing(self, reset=True):
        ms = np.zeros(4)
        n = np.zeros(4, np.int64)
        self._chk(self.lib.ilqgb_timing(self.h, _ptr(ms), _ptr(n), int(reset)))
        return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(KERNEL_CLASSES)}
