"""Host-side engine: device-resident environment batch, actor sampler, GAE and RK4 entry points.

Everything here is plumbing around libsatb200.so (include/satb200.h): torch allocates device memory
and provides the stream; all arithmetic of the hot path runs in the CUDA kernels. There is no CPU
fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import math

import numpy as np

from . import _lib as L

# physical constants of the reference
MU_KM, RE_KM, J2 = 398600.0, 6378.137, 0.00108263          # RK4 script :9-11
MU_M, RE_M = 3.986e14, 6378137.0                           # satellite_function.py:28
OBS_DIM, ACT_DIM = 18, 3


def cw_stm(t: float = 100.0) -> np.ndarray:
    """6x6 Clohessy-Wiltshire state-transition matrix exactly as the reference builds it
    (satellite_function.py:753-773): python-float omega/tau, numpy sin/cos."""
    u = 3.986e14
    R = 42164000
    omega = math.sqrt(u / (R ** 3))
    tau = omega * t
    s = np.sin(tau)
    c = np.cos(tau)
    return np.array([
        [4 - 3 * c, 0, 0, s / omega, 2 * (1 - c) / omega, 0],
        [6 * (s - tau), 1, 0, -2 * (1 - c) / omega, 4 * s / omega - 3 * tau, 0],
        [0, 0, c, 0, 0, s / omega],
        [3 * omega * s, 0, 0, c, 2 * s, 0],
        [6 * omega * (c - 1), 0, 0, -2 * s, 4 * c - 3, 0],
        [0, 0, -omega * s, 0, 0, c]], dtype=np.float64)


def _round_up(n: int, m: int) -> int:
    return (n + m - 1) // m * m


# --------------------------------------------------------------------------------------------- K1
def rk4_propagate(x, h: float, substeps: int, mu: float = MU_KM, re: float = RE_KM, j2: float = J2):
    """In-place RK4 propagation of a CUDA fp64 tensor x [6, N] (rows x,y,z,vx,vy,vz).
    Replaces `substeps` calls of RungeKutta (RK4 script :34-40) per state."""
    torch = L.require_cuda()
    if x.dtype != torch.float64 or x.dim() != 2 or x.shape[0] != 6:
        raise L.SatError("x must be a float64 CUDA tensor of shape [6, N]")
    n, ld = x.shape[1], x.stride(0)
    if x.stride(1) != 1:
        raise L.SatError("x rows must be contiguous")
    L.check(L.load().sat_rk4_propagate(x.data_ptr(), n, ld, float(h), int(substeps), float(mu), float(re),
                                       float(j2), L.stream_ptr()), "sat_rk4_propagate")
    return x


def alloc_soa(rows: int, n: int, dtype, device):
    """[rows, n] view of a buffer whose row stride is even and 16-byte aligned (vector loads)."""
    torch = L.require_cuda()
    ld = _round_up(n, 2)
    buf = torch.zeros((rows, ld), dtype=dtype, device=device)
    return buf[:, :n], buf


class Rk4HostPropagator:
    """Host-buffer form (numpy in / numpy out through pinned staging): the e2e path of K1."""

    def __init__(self, n: int, device="cuda"):
        torch = L.require_cuda()
        self.n = n
        self.ld = _round_up(n, 2)
        self.dev = torch.empty((6, self.ld), dtype=torch.float64, device=device)
        self.pinned = torch.empty((6, n), dtype=torch.float64).pin_memory()

    def __call__(self, x_np: np.ndarray, h, substeps, mu=MU_KM, re=RE_KM, j2=J2) -> np.ndarray:
        self.pinned.numpy()[...] = x_np
        L.check(L.load().sat_rk4_propagate_host(self.pinned.data_ptr(), self.n, self.dev.data_ptr(), self.ld,
                                                float(h), int(substeps), float(mu), float(re), float(j2),
                                                L.stream_ptr()), "sat_rk4_propagate_host")
        return self.pinned.numpy().copy()


# --------------------------------------------------------------------------------------------- stats
class RunningStats:
    """Device-resident RunningMeanStd (normalization.py:7-29): [n | mean[dim] | S[dim] | std[dim]]."""

    def __init__(self, dim: int, device="cuda"):
        torch = L.require_cuda()
        self.dim = dim
        self.buf = torch.zeros(1 + 3 * dim, dtype=torch.float64, device=device)

    @property
    def n(self):
        return int(self.buf[0].item())

    @property
    def mean(self):
        return self.buf[1:1 + self.dim]

    @property
    def S(self):
        return self.buf[1 + self.dim:1 + 2 * self.dim]

    @property
    def std(self):
        return self.buf[1 + 2 * self.dim:1 + 3 * self.dim]

    def state_dict(self):
        return {"dim": self.dim, "buf": self.buf.detach().cpu().clone()}

    def load_state_dict(self, sd):
        assert int(sd["dim"]) == self.dim
        self.buf.copy_(sd["buf"].to(self.buf.device))
        return self

    def update_normalize(self, x, update=True, out_dtype=None, group=None):
        """x: CUDA fp64 [n, dim]. Merges the batch (update=True) then returns (x-mean)/(std+1e-8).
        group (a torch.distributed process group): x is this rank's shard of a batch sharded over the group, and the
        merge folds every rank's shard (sat_stats_fold), so every rank's statistics become those of the union batch - bit
        for bit when every rank but the last brings a multiple of 128 rows. Collective: every rank of the group calls it."""
        torch = L.require_cuda()
        lib = L.load()
        x = x.contiguous()
        n = x.shape[0]
        ws = torch.empty(lib.sat_workspace_bytes(n), dtype=torch.uint8, device=x.device)
        if update and group is not None:
            ex = StatsExchange(group, n, self.dim, x.device)
            L.check(lib.sat_norm_partials(L.ptr(x), n, self.dim, L.ptr(ex.send), ws.data_ptr(), L.stream_ptr()),
                    "sat_norm_partials")
            ex.fold(self, None, None, ws)
            update = False
        out64 = torch.empty_like(x) if out_dtype in (None, torch.float64) else None
        out32 = torch.empty(x.shape, dtype=torch.float32, device=x.device) if out_dtype == torch.float32 else None
        L.check(lib.sat_norm_update(self.buf.data_ptr(), x.data_ptr(), n, self.dim, int(bool(update)),
                                    L.ptr(out64), L.ptr(out32), ws.data_ptr(), L.stream_ptr()),
                "sat_norm_update")
        return out64 if out64 is not None else out32


def fold_stats(partials, rank_rows, dim: int, obs_stats: RunningStats | None = None, ret_stats: RunningStats | None = None,
               ret_std_out=None, workspace=None):
    """sat_stats_fold: fold the gathered per-block partials of G ranks into the statistics.
    partials: CUDA fp64 [G, stride] rank-major, each row one rank's partials padded to a common length; rank_rows: CUDA
    int64 [G] row counts. dim 0: env-step partials (EnvBatch.step_partials) into obs_stats (18) / ret_stats (1) /
    ret_std_out; dim >= 1: sat_norm_partials of a [n, dim] batch into obs_stats. workspace: the workspace the partials were
    just computed with on this stream (its ticket is zero)."""
    torch = L.require_cuda()
    dims = 19 if dim == 0 else dim
    if partials.dtype != torch.float64 or partials.dim() != 2 or partials.shape[1] % (2 * dims):
        raise L.SatError(f"partials must be float64 [ranks, blocks * {2 * dims}]")
    if rank_rows.dtype != torch.int64 or rank_rows.numel() != partials.shape[0]:
        raise L.SatError("rank_rows must be int64 with one row count per rank")
    L.check(L.load().sat_stats_fold(L.ptr(partials), partials.shape[0], partials.shape[1] // (2 * dims), L.ptr(rank_rows),
                                    int(dim), L.ptr(obs_stats.buf) if obs_stats is not None else None,
                                    L.ptr(ret_stats.buf) if ret_stats is not None else None, L.ptr(ret_std_out),
                                    L.ptr(workspace), L.stream_ptr()), "sat_stats_fold")


class StatsExchange:
    """Per-block statistics partials exchanged across the ranks of a process group: `send` takes this rank's partials,
    fold() gathers every rank's (torch.distributed.all_gather_into_tensor on the current stream; NCCL or gloo) into one
    rank-major buffer and folds them all into this rank's statistics (sat_stats_fold), so every rank holds the same bits.
    dim 0: the env step's partials (64 rows per block, 19 dims); dim >= 1: a [rows, dim] batch's (128 rows per block).

    Construction is collective: every rank's (rows, dim) are gathered once and checked by every rank on the same data, so
    either every rank proceeds or every rank raises."""

    def __init__(self, group, rows: int, dim: int, device):
        torch = L.require_cuda()
        dist = torch.distributed
        self.group, self.dim = group, int(dim)
        world = dist.get_world_size(group)
        mine = torch.tensor([int(rows), int(dim)], dtype=torch.int64, device=device)
        every = torch.empty(world * 2, dtype=torch.int64, device=device)
        dist.all_gather_into_tensor(every, mine, group=group)
        every = every.view(world, 2).cpu()
        rows_all, dims_all = every[:, 0].tolist(), every[:, 1].tolist()
        if len(set(dims_all)) != 1 or min(rows_all) < 1:
            raise L.SatError(f"shared statistics need the same dim and at least one row on every rank; got rows {rows_all}, "
                             f"dims {dims_all}")
        rpb = 64 if dim == 0 else 128
        dims = 19 if dim == 0 else dim
        stride = max((r + rpb - 1) // rpb for r in rows_all)
        self.rank_rows = every[:, 0].to(device).contiguous()
        self.send = torch.zeros(stride * dims * 2, dtype=torch.float64, device=device)
        self.gathered = torch.zeros((world, stride * dims * 2), dtype=torch.float64, device=device)

    def fold(self, obs_stats: RunningStats | None, ret_stats: RunningStats | None, ret_std_out, workspace):
        """gather every rank's `send` and fold them all; workspace as for fold_stats"""
        import torch.distributed as dist
        dist.all_gather_into_tensor(self.gathered.view(-1), self.send, group=self.group)
        fold_stats(self.gathered, self.rank_rows, self.dim, obs_stats, ret_stats, ret_std_out, workspace)


# --------------------------------------------------------------------------------------------- K2
class EnvBatch:
    """N independent `satellites` environments resident on one GPU (SoA fp64 state, int32 counters).

    mode "cw": the env as shipped (CW STM, environment.py:117-121) -> bit-level parity target.
    mode "rk4": propagation by `substeps` RK4 steps of size h of the inertial two-body+J2 ODE
    (north-star production path; relative<->inertial by the reference's translation, environment.py:334-343).

    start_box=(lo, hi), two length-12 sequences over (P, Pv, E, Ev) in the CW frame (metres, m/s): starts mode. Every env
    owns a start, drawn on the device uniformly in lo <= x <= hi (lo == hi fixes a column) and keyed by (start_seed,
    row_offset + env index, draw index) only, so a sharded batch or a resumed run draws the same starts. Every reset of an
    env, manual or automatic, puts its kinematics at its start (count 0, int_state 0; fuel / dis / dangerous_zone persist)
    and then draws its next one. `starts` is the [12, n] view of the next starts. start_box=None: the reference's reset
    literals for every env.

    share_stats(group): the batch is one rank's shard of a batch sharded over a process group, and step() updates its
    running statistics with every rank's shard (see share_stats).
    """

    def __init__(self, n: int, mode: str = "cw", flag: int = 0, d_capture: float = 100000.0,
                 d_range: float = 100000.0, fuel_c: float = 320.0, fuel_t: float = 320.0,
                 max_episode_steps: int = 1000, auto_reset: bool = True, substeps: int = 100, h: float = 1.0,
                 j2: float = J2, gamma: float = 0.99, skip_danger_zone: bool = False, t_step: float = 100.0,
                 fast_libm: bool = False,
                 stm: np.ndarray | None = None, device="cuda", start_box=None, start_seed: int = 0, row_offset: int = 0):
        torch = L.require_cuda()
        self.torch = torch
        self.lib = L.load()
        self.n = int(n)
        self.device = torch.device(device)
        self.start_box = None if start_box is None else _start_box(start_box)
        self.start_seed, self.row_offset, self.start_draws = int(start_seed) & (2 ** 64 - 1), int(row_offset), 0
        if self.row_offset < 0:
            raise L.SatError("row_offset must be >= 0")
        cols = L.SAT_STATE_COLS if self.start_box is None else L.SAT_STATE_COLS_STARTS
        self.state, self._state_buf = alloc_soa(cols, self.n, torch.float64, self.device)
        self.istate, self._istate_buf = alloc_soa(L.SAT_ISTATE_COLS, self.n, torch.int32, self.device)
        self.ld = self._state_buf.shape[1]
        self.st = L.SatEnvState(self._state_buf.data_ptr(), self._istate_buf.data_ptr(), self.n, self.ld)
        p = L.default_params()
        p.mode = {"cw": L.MODE_CW, "rk4": L.MODE_RK4}[mode]
        p.flag = int(flag)
        p.max_episode_steps = int(max_episode_steps)
        p.auto_reset = (1 if self.start_box is None else L.RESET_STARTS) if auto_reset else 0
        p.substeps = int(substeps)
        p.skip_danger_zone = int(bool(skip_danger_zone))
        p.fast_libm = int(bool(fast_libm))        # False: exact host-libm arithmetic in the danger-zone count (bit parity)
        p.d_capture, p.d_range, p.gamma = float(d_capture), float(d_range), float(gamma)
        p.h, p.j2 = float(h), float(j2)
        M = cw_stm(t_step) if stm is None else np.asarray(stm, dtype=np.float64)
        for i, v in enumerate(M.ravel()):
            p.stm[i] = float(v)
        self.params = p
        self.mode = mode
        self._fuel0 = (float(fuel_c), float(fuel_t))
        self.workspace = torch.empty(self.lib.sat_workspace_bytes(self.n), dtype=torch.uint8, device=self.device)
        self.reward = torch.empty(self.n, dtype=torch.float64, device=self.device)
        self.done = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        self._host = None
        self._shared = None
        self.init()

    # -- parameters that the reference lets the driver patch after construction (CPPO_main.py:98)
    @property
    def d_capture(self):
        return self.params.d_capture

    @d_capture.setter
    def d_capture(self, v):
        self.params.d_capture = float(v)

    def init(self):
        """constructor state + reset() (environment.py:26-62, 66-79). Starts mode: then every env's first start is drawn,
        the envs are reset to it, and every env's next start is drawn."""
        L.guard_device(self.device)
        L.check(self.lib.sat_env_init(C.byref(self.st), self._fuel0[0], self._fuel0[1], C.byref(self.params),
                                      L.stream_ptr()), "sat_env_init")
        if self.start_box is not None:
            self.draw_starts()
            L.check(self.lib.sat_env_reset_starts(C.byref(self.st), None, L.stream_ptr()), "sat_env_reset_starts")
            self.draw_starts()

    def reset(self, mask=None, flag=None):
        """reset(Flag) for the masked envs (uint8 CUDA tensor) or all; fuel/dis/dangerous_zone persist (Q2).
        Starts mode: the masked envs go to their starts (count 0, int_state 0), then their next starts are drawn."""
        if flag is not None:
            self.params.flag = int(flag)
        if self.start_box is not None:
            L.check(self.lib.sat_env_reset_starts(C.byref(self.st), L.ptr(mask), L.stream_ptr()), "sat_env_reset_starts")
            self.draw_starts(mask)
            return
        L.check(self.lib.sat_env_reset(C.byref(self.st), L.ptr(mask), C.byref(self.params), L.stream_ptr()),
                "sat_env_reset")

    def draw_starts(self, mask=None):
        """draw the next start of the masked envs (uint8 CUDA tensor; None = all) into the start columns; one draw index
        (start_draws) per call"""
        if self.start_box is None:
            raise L.SatError("draw_starts needs a batch built with start_box")
        L.guard_device(self.device)
        lo, hi = self.start_box
        L.check(self.lib.sat_env_draw_starts(C.byref(self.st), L.ptr(mask), (C.c_double * 12)(*lo), (C.c_double * 12)(*hi),
                                             self.start_seed, self.start_draws & 0xFFFFFFFF, self.row_offset,
                                             L.stream_ptr()), "sat_env_draw_starts")
        self.start_draws += 1

    @property
    def starts(self):
        """[12, n] view of every env's next start (columns P, Pv, E, Ev); None without start_box"""
        return None if self.start_box is None else self.state[L.COL_START:L.COL_START + 12]

    def _redraw_after_step(self, done):
        # the step reset its finished envs to their starts (same launch); they now need their next ones
        if self.start_box is not None and self.params.auto_reset == L.RESET_STARTS:
            self.draw_starts(done)

    def observe(self, dtype=None):
        torch = self.torch
        dtype = dtype or torch.float64
        out = torch.empty((self.n, OBS_DIM), dtype=dtype, device=self.device)
        L.check(self.lib.sat_env_observe(C.byref(self.st), L.ptr(out) if dtype == torch.float32 else None,
                                         L.ptr(out) if dtype == torch.float64 else None, L.stream_ptr()),
                "sat_env_observe")
        return out

    def step(self, pa, ea, count=None, obs_f32=None, obs_f64=None, term_obs_f64=None, reward=None, done=None,
             obs_stats: RunningStats | None = None, ret_stats: RunningStats | None = None, ret_std_out=None):
        """One step() of every env. pa/ea: CUDA [n,3] float32 or float64. Outputs are written into the
        given tensors (allocated by the caller to keep the hot loop allocation-free). After share_stats(group), the
        statistics are updated with every rank's step (collective)."""
        torch = self.torch
        if self._shared is not None and (obs_stats is not None or ret_stats is not None):
            reward, done = self.step_partials(pa, ea, self._shared.send, count, obs_f32, obs_f64, term_obs_f64, reward,
                                              done)
            self._shared.fold(obs_stats, ret_stats, ret_std_out, self.workspace)
            return reward, done
        L.guard_device(self.device)
        if pa.dtype != ea.dtype or pa.dtype not in (torch.float32, torch.float64):
            raise L.SatError("actions must both be float32 or both float64")
        self.params.action_dtype = L.ACT_F32 if pa.dtype == torch.float32 else L.ACT_F64
        reward = self.reward if reward is None else reward
        done = self.done if done is None else done
        L.check(self.lib.sat_env_step(C.byref(self.st), L.ptr(pa), L.ptr(ea), L.ptr(count), L.ptr(obs_f32),
                                      L.ptr(obs_f64), L.ptr(term_obs_f64), L.ptr(reward), L.ptr(done),
                                      L.ptr(obs_stats.buf) if obs_stats is not None else None,
                                      L.ptr(ret_stats.buf) if ret_stats is not None else None,
                                      L.ptr(ret_std_out), self.workspace.data_ptr(), C.byref(self.params),
                                      L.stream_ptr()), "sat_env_step")
        self._redraw_after_step(done)
        return reward, done

    def share_stats(self, group):
        """Shared-statistics mode: from now on step() with obs_stats / ret_stats folds the statistics partials of every
        rank of `group` (a torch.distributed process group, each rank holding its shard of the envs) into this rank's
        statistics: step with the partials out (sat_env_step_partials), all_gather them, fold them all (sat_stats_fold).
        Every rank then holds the same statistics, bit-identical to one batch of the union of the shards stepping the
        union of the actions whenever every rank but the last holds a multiple of 64 envs (and row_offset / start_seed
        key each env by its global index). Collective: every rank calls it, and every rank's step() must then pass the
        same set of statistics. group=None switches back to per-rank statistics (not collective)."""
        self._shared = None if group is None else StatsExchange(group, self.n, 0, self.device)
        return self

    def step_partials(self, pa, ea, partials, count=None, obs_f32=None, obs_f64=None, term_obs_f64=None, reward=None,
                      done=None):
        """step() with statistics on, but the per-block partials go to `partials` (CUDA fp64, at least
        sat_stats_partials_bytes(n, 0) bytes) instead of into any statistics; fold_stats() folds them. The workspace
        of this batch is then ready for fold_stats()."""
        torch = self.torch
        L.guard_device(self.device)
        if pa.dtype != ea.dtype or pa.dtype not in (torch.float32, torch.float64):
            raise L.SatError("actions must both be float32 or both float64")
        if partials.dtype != torch.float64 or partials.numel() * 8 < self.lib.sat_stats_partials_bytes(self.n, 0):
            raise L.SatError("partials must be float64 of at least sat_stats_partials_bytes(n, 0) bytes")
        self.params.action_dtype = L.ACT_F32 if pa.dtype == torch.float32 else L.ACT_F64
        reward = self.reward if reward is None else reward
        done = self.done if done is None else done
        L.check(self.lib.sat_env_step_partials(C.byref(self.st), L.ptr(pa), L.ptr(ea), L.ptr(count), L.ptr(obs_f32),
                                               L.ptr(obs_f64), L.ptr(term_obs_f64), L.ptr(reward), L.ptr(done),
                                               L.ptr(partials), self.workspace.data_ptr(), C.byref(self.params),
                                               L.stream_ptr()), "sat_env_step_partials")
        self._redraw_after_step(done)
        return reward, done

    def step_timed(self, pa, ea, reward=None, done=None, obs_stats: RunningStats | None = None,
                   ret_stats: RunningStats | None = None):
        """step() through sat_env_step_timed: returns (front_ms, finish_ms, merge_ms) measured with CUDA events recorded
        between the launches on the launching stream (bench.py's per-kernel roofline)."""
        self.params.action_dtype = L.ACT_F32 if pa.dtype == self.torch.float32 else L.ACT_F64
        ms = (C.c_float * 3)()
        done = self.done if done is None else done
        L.check(self.lib.sat_env_step_timed(C.byref(self.st), L.ptr(pa), L.ptr(ea), None, None, None, None,
                                            L.ptr(self.reward if reward is None else reward), L.ptr(done),
                                            L.ptr(obs_stats.buf) if obs_stats is not None else None,
                                            L.ptr(ret_stats.buf) if ret_stats is not None else None, None,
                                            self.workspace.data_ptr(), C.byref(self.params), L.stream_ptr(), ms),
                "sat_env_step_timed")
        self._redraw_after_step(done)
        return float(ms[0]), float(ms[1]), float(ms[2])

    # -- host-buffer form: the reference-facing call with numpy in / numpy out (e2e path)
    def host_buffers(self):
        """pinned host arrays (pa, ea, obs, reward, done). Filling pa/ea in place and passing them to step_host()
        avoids the staging memcpy; obs/reward/done are overwritten by every step_host() call."""
        torch = self.torch
        if self._host is None:
            n = self.n
            self._host = dict(
                pa=torch.empty((n, 3), dtype=torch.float32).pin_memory(),
                ea=torch.empty((n, 3), dtype=torch.float32).pin_memory(),
                obs=torch.empty((n, OBS_DIM), dtype=torch.float32).pin_memory(),
                rew=torch.empty(n, dtype=torch.float64).pin_memory(),
                done=torch.empty(n, dtype=torch.uint8).pin_memory(),
                dio=torch.zeros(self.lib.sat_env_step_host_bytes(n), dtype=torch.uint8, device=self.device),
                aux_stream=torch.cuda.Stream(device=self.device))
            hb = self._host
            hb["np"] = tuple(hb[k].numpy() for k in ("pa", "ea", "obs", "rew", "done"))
        return self._host["np"]

    def step_host(self, pa_np: np.ndarray, ea_np: np.ndarray):
        """step(pa, ea) with HOST arrays in and out: one sat_env_step_host call on the pinned host arrays, which the
        kernels read and write directly (UVA zero-copy). In rk4 mode the propagation kernel also emits the next
        observation, which a copy engine moves to the host on a second stream underneath the danger-zone kernel:
        241 us/step at 65 536 envs on a B200 (DESIGN.md s6c has the forms measured before it). Returns pinned numpy views
        (valid until the next call)."""
        pa_h, ea_h, obs_h, rew_h, done_h = self.host_buffers()
        hb = self._host
        if pa_np is not pa_h:
            pa_h[...] = pa_np
        if ea_np is not ea_h:
            ea_h[...] = ea_np
        L.check(self.lib.sat_env_step_host(C.byref(self.st), hb["pa"].data_ptr(), hb["ea"].data_ptr(),
                                           hb["obs"].data_ptr(), hb["rew"].data_ptr(), hb["done"].data_ptr(),
                                           hb["dio"].data_ptr(), C.byref(self.params), L.stream_ptr(),
                                           hb["aux_stream"].cuda_stream),
                "sat_env_step_host")
        if self.start_box is not None and self.params.auto_reset == L.RESET_STARTS:
            self.done.copy_(hb["done"])                      # the step synchronised: done_h is final
            self._redraw_after_step(self.done)
        return obs_h, rew_h, done_h

    @property
    def h2d_bytes_per_step(self):
        return self.n * 3 * 4 * 2

    @property
    def d2h_bytes_per_step(self):
        return self.n * (OBS_DIM * 4 + 8 + 1)

    # -- checkpoint / resume of the full environment state (the reference saves only the networks, SURVEY s5)
    def state_dict(self):
        p = self.params
        return {"n": self.n, "mode": self.mode, "state": self.state.detach().cpu().clone(),
                "istate": self.istate.detach().cpu().clone(),
                "start_box": self.start_box, "start_seed": self.start_seed, "row_offset": self.row_offset,
                "start_draws": self.start_draws,
                "params": {k: (list(getattr(p, k)) if hasattr(getattr(p, k), "__len__") else getattr(p, k))
                           for k, _t in p._fields_}}

    def load_state_dict(self, sd):
        if int(sd["n"]) != self.n or sd["mode"] != self.mode:
            raise L.SatError("checkpoint is for a different batch size / propagation mode")
        if (sd.get("start_box") is None) != (self.start_box is None):
            raise L.SatError("checkpoint is for a batch %s start_box" % ("without" if self.start_box is not None else "with"))
        if self.start_box is not None:
            self.start_box = _start_box(sd["start_box"])
            self.start_seed, self.row_offset = int(sd["start_seed"]), int(sd["row_offset"])
            self.start_draws = int(sd["start_draws"])
        self.state.copy_(sd["state"].to(self.device))
        self.istate.copy_(sd["istate"].to(self.device))
        for k, v in sd["params"].items():
            if isinstance(v, list):
                arr = getattr(self.params, k)
                for i, x in enumerate(v):
                    arr[i] = x
            else:
                setattr(self.params, k, v)
        return self

    # -- convenient views (fp64, exact)
    def positions(self):
        s = self.state
        return s[0:3].T, s[3:6].T, s[6:9].T, s[9:12].T

    def set_state(self, P, Pv, E, Ev):
        """overwrite the 12 kinematic columns (tensors/arrays [n,3]); clears the int64 quirk flag."""
        torch = self.torch
        for off, a in ((0, P), (3, Pv), (6, E), (9, Ev)):
            self.state[off:off + 3] = torch.as_tensor(np.asarray(a, dtype=np.float64), device=self.device).T
        self.istate[L.ICOL_INTSTATE].zero_()

    @property
    def fuel_c(self):
        return self.state[L.COL_FUEL_C]

    @property
    def fuel_t(self):
        return self.state[L.COL_FUEL_T]

    @property
    def dis(self):
        return self.state[L.COL_DIS]

    @property
    def dangerous_zone(self):
        return self.istate[L.ICOL_DZ]

    @property
    def episode_count(self):
        return self.istate[L.ICOL_COUNT]

    @property
    def err(self):
        return self.istate[L.ICOL_ERR]


def _start_box(box):
    """(lo, hi) -> two 12-tuples of floats, lo <= hi, all finite"""
    try:
        lo, hi = box
        lo, hi = tuple(float(x) for x in np.asarray(lo, dtype=np.float64).ravel()), \
            tuple(float(x) for x in np.asarray(hi, dtype=np.float64).ravel())
    except (TypeError, ValueError) as exc:
        raise L.SatError("start_box must be (lo, hi), two sequences of 12 numbers") from exc
    if len(lo) != 12 or len(hi) != 12:
        raise L.SatError("start_box must be (lo, hi), two sequences of 12 numbers (P, Pv, E, Ev)")
    if not all(math.isfinite(a) and math.isfinite(b) and a <= b and math.isfinite(b - a) for a, b in zip(lo, hi)):
        raise L.SatError("start_box needs finite bounds with lo <= hi")
    return lo, hi


def danger_zone_count(rv, dv, u=MU_M, debug=False):
    """Batched Time_window_of_danger_zone(...).calculate_number_of_hanger_area() (satellite_function.py:341-373).
    rv: CUDA fp64 [n,12] = (R0_c, V0_c, R0_t, V0_t) inertial, metres; dv: [n] Delta_V_c. -> int32 [n]."""
    torch = L.require_cuda()
    rv, dv = rv.contiguous(), dv.contiguous()
    n = rv.shape[0]
    out = torch.empty(n, dtype=torch.int32, device=rv.device)
    dbg = torch.zeros((n, 2, 8), dtype=torch.float64, device=rv.device) if debug else None
    L.check(L.load().sat_danger_zone_count(L.ptr(rv), L.ptr(dv), n, float(u), L.ptr(out), L.ptr(dbg), L.stream_ptr()),
            "sat_danger_zone_count")
    return (out, dbg) if debug else out


def numerical_iteration(dvm, theta, v1x, v1y, h, guess, u=MU_M, return_nfev=False):
    """Batched Time_window_of_danger_zone.Numerical_iteration_method (satellite_function.py:558-565): one
    scipy.optimize.fsolve root of P_fai_equation per element. CUDA fp64 [n] arrays -> roots [n] (un-polished result[0])."""
    torch = L.require_cuda()
    args = [a.contiguous() for a in (dvm, theta, v1x, v1y, h, guess)]
    n = args[0].shape[0]
    root = torch.empty(n, dtype=torch.float64, device=args[0].device)
    nfev = torch.empty(n, dtype=torch.int32, device=args[0].device) if return_nfev else None
    L.check(L.load().sat_fsolve_pfai(*[L.ptr(a) for a in args], n, float(u), L.ptr(root), L.ptr(nfev), L.stream_ptr()),
            "sat_fsolve_pfai")
    return (root, nfev) if return_nfev else root


LIBM_FN = {"sin": 0, "cos": 1, "acos": 2, "atan": 3, "pow2": 4, "sincos_s": 5, "sincos_c": 6}


def libm_eval(fn: str, x):
    """The device libm of the danger-zone path (csrc/glibm.cuh: numpy scalar sin / cos / arccos / arctan, python x ** 2)
    evaluated elementwise on a CUDA fp64 tensor; exists so tests can compare it bit for bit with the host libm."""
    torch = L.require_cuda()
    x = x.contiguous()
    y = torch.empty_like(x)
    L.check(L.load().sat_libm_eval(LIBM_FN[fn], L.ptr(x), L.ptr(y), x.numel(), L.stream_ptr()), "sat_libm_eval")
    return y


def reachable_domain(elements, delta_max, N2=200, N3=200, u=MU_M):
    """Batched RD_single_pulse.Reachable_Domain sweep. elements: CUDA fp64 [n,6] (a,e,i,omega,Omega,f); delta_max [n].
    -> rf_max [n,D,3], rf_min [n,D,3], valid [n,D] (uint8), D = (N2+1)*(N3+1) directions in the reference's loop order."""
    torch = L.require_cuda()
    elements, delta_max = elements.contiguous(), delta_max.contiguous()
    n = elements.shape[0]
    D = (N2 + 1) * (N3 + 1)
    hi = torch.empty((n, D, 3), dtype=torch.float64, device=elements.device)
    lo = torch.empty((n, D, 3), dtype=torch.float64, device=elements.device)
    valid = torch.empty((n, D), dtype=torch.uint8, device=elements.device)
    L.check(L.load().sat_reachable_domain(L.ptr(elements), L.ptr(delta_max), n, int(N2), int(N3), float(u), L.ptr(hi),
                                          L.ptr(lo), L.ptr(valid), L.stream_ptr()), "sat_reachable_domain")
    return hi, lo, valid


# --------------------------------------------------------------------------------------------- K3
class GaussianActorKernel:
    """Fused Actor_Gaussian forward + sampling (ppo_continuous.py:83-95, 176-189) for batches."""

    KEYS = ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "mean_layer.weight", "mean_layer.bias", "log_std")

    def __init__(self, max_action: float = 1.6, use_tanh: bool = True, device="cuda", critic: bool = False):
        torch = L.require_cuda()
        self.torch = torch
        self.lib = L.load()
        self.device = torch.device(device)
        self.critic = critic
        self.packed = torch.zeros(L.ACTOR_PACKED_FLOATS, dtype=torch.float32, device=self.device)
        self.max_action = float(max_action)
        self.use_tanh = int(bool(use_tanh))
        self._keep = None
        self.w = None
        # both dense layers on the tensor cores (exact bf16x3 split, csrc/actor_tc.cu): the default; SAT_ACTOR_TC=0 or
        # sample(tc=False) selects the fp32 FFMA2 kernel (csrc/actor.cu)
        self.use_tc = os.environ.get("SAT_ACTOR_TC", "1") == "1"
        self._tc_image = None

    def load_state_dict(self, sd):
        """sd: torch state_dict (or dict of arrays) with the reference's parameter names."""
        torch = self.torch
        names = (("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias") if self.critic
                 else self.KEYS[:6])
        t = [torch.as_tensor(np.asarray(sd[k].detach().cpu() if hasattr(sd[k], "detach") else sd[k]),
                             dtype=torch.float32).contiguous().to(self.device) for k in names]
        if self.critic:
            ls = None
        else:
            v = sd["log_std"]
            ls = torch.as_tensor(np.asarray(v.detach().cpu() if hasattr(v, "detach") else v),
                                 dtype=torch.float32).reshape(-1).contiguous().to(self.device)
        hid, in_dim = t[0].shape
        heads = t[4].shape[0]
        w = L.SatActorWeights(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), t[4].data_ptr(),
                              t[5].data_ptr(), ls.data_ptr() if ls is not None else None, self.packed.data_ptr(),
                              in_dim, hid, heads, self.use_tanh, self.max_action)
        L.check(self.lib.sat_actor_pack(C.byref(w), self.packed.data_ptr(), L.stream_ptr()), "sat_actor_pack")
        self._keep = (t, ls)
        self.w = w
        return self

    def sample(self, obs=None, env: EnvBatch | None = None, obs_stats: RunningStats | None = None, seed: int = 0,
               step: int = 0, row_offset: int = 0, eps_in=None, act=None, logp=None, mean_out=None, eps_out=None,
               obs_out=None, tc: bool | None = None):
        """obs: CUDA fp32 [n,18]; or env=EnvBatch to read (and optionally normalise) the state directly.
        tc: run the dense layers as bf16x3 on the tensor cores (sat_actor_sample_tc); default = self.use_tc."""
        torch = self.torch
        L.guard_device(self.device)
        if self.w is None:
            raise L.SatError("weights not loaded")
        n = obs.shape[0] if obs is not None else env.n
        act = torch.empty((n, ACT_DIM), dtype=torch.float32, device=self.device) if act is None else act
        logp = torch.empty((n, ACT_DIM), dtype=torch.float32, device=self.device) if logp is None else logp
        if (self.use_tc if tc is None else tc) and not self.critic:
            if obs is None:
                obs, env, obs_stats, obs_out = self._tc_obs(env, obs_stats, obs_out), None, None, None
            L.check(self.lib.sat_actor_sample_tc(C.byref(self.w), self._image().data_ptr(), L.ptr(obs),
                                                 C.byref(env.st) if env is not None else None,
                                                 L.ptr(obs_stats.buf) if obs_stats is not None else None, n,
                                                 int(row_offset), int(seed) & (2 ** 64 - 1), int(step) & (2 ** 64 - 1),
                                                 L.ptr(eps_in), L.ptr(act), L.ptr(logp), L.ptr(mean_out), L.ptr(eps_out),
                                                 L.ptr(obs_out), L.stream_ptr()), "sat_actor_sample_tc")
            return act, logp
        L.check(self.lib.sat_actor_sample(C.byref(self.w), L.ptr(obs), C.byref(env.st) if env is not None else None,
                                          L.ptr(obs_stats.buf) if obs_stats is not None else None, n,
                                          int(row_offset), int(seed) & (2 ** 64 - 1), int(step) & (2 ** 64 - 1),
                                          L.ptr(eps_in), L.ptr(act), L.ptr(logp), L.ptr(mean_out), L.ptr(eps_out),
                                          L.ptr(obs_out), L.stream_ptr()), "sat_actor_sample")
        return act, logp

    def _tc_obs(self, env, obs_stats, obs_out):
        """tensor-core path on the env state: the fp32 (normalised) observation is materialised by one streaming kernel
        (sat_env_observe_norm, the fused path's arithmetic) into obs_out / a cached scratch and the GEMM kernel reads that:
        rebuilding it inside the kernel cost the row warps 4.6 us per 128-row tile (fp64 loads + divisions on 8 of 16 warps)."""
        n = env.n
        if obs_out is None:
            if getattr(self, "_obs_scratch", None) is None or self._obs_scratch.shape[0] < n:
                self._obs_scratch = self.torch.empty((n, OBS_DIM), dtype=self.torch.float32, device=self.device)
            obs_out = self._obs_scratch[:n]
        L.check(self.lib.sat_env_observe_norm(C.byref(env.st), L.ptr(obs_stats.buf) if obs_stats is not None else None,
                                              L.ptr(obs_out), L.stream_ptr()), "sat_env_observe_norm")
        return obs_out

    def _image(self):
        if self._tc_image is None:
            self._tc_image = self.torch.empty(L.ACTOR_TC_IMAGE_FLOATS, dtype=self.torch.float32, device=self.device)
        return self._tc_image

    def sample_pair(self, other, obs=None, env: EnvBatch | None = None, obs_stats: RunningStats | None = None,
                    seed: int = 0, step: int = 0, other_step: int = 1, row_offset: int = 0, act=None, logp=None,
                    obs_out=None, other_act=None, other_logp=None, tc: bool | None = None):
        """this actor and `other` on the same observations: exactly self.sample(step=step) and
        other.sample(step=other_step) -> (act, logp, other_act, other_logp). Tensor-core path (default): both networks' row
        tiles go through ONE persistent grid (sat_actor_sample_pair_tc) at any batch size. FFMA2 path (tc=False): up to 32 768
        rows both networks go into one launch (sat_actor_sample_pair) so that they share the GPU - measured one-launch /
        two-launch times: 4096 rows 44 / 75 us, 8192: 66 / 76, 32 768: 201 / 222; at 65 536 rows each network fills the GPU
        by itself (388 / 374) and two launches are issued."""
        torch = self.torch
        L.guard_device(self.device)
        if self.w is None or other.w is None:
            raise L.SatError("weights not loaded")
        n = obs.shape[0] if obs is not None else env.n
        use_tc = (self.use_tc if tc is None else tc) and not self.critic and not other.critic and self.use_tanh == other.use_tanh
        if n > 32768 and not use_tc:
            act, logp = self.sample(obs=obs, env=env, obs_stats=obs_stats, seed=seed, step=step, row_offset=row_offset,
                                    act=act, logp=logp, obs_out=obs_out, tc=False)
            other_act, other_logp = other.sample(obs=obs, env=env, obs_stats=obs_stats, seed=seed, step=other_step,
                                                 row_offset=row_offset, act=other_act, logp=other_logp, tc=False)
            return act, logp, other_act, other_logp
        new = lambda: torch.empty((n, ACT_DIM), dtype=torch.float32, device=self.device)
        act = new() if act is None else act
        logp = new() if logp is None else logp
        other_act = new() if other_act is None else other_act
        other_logp = new() if other_logp is None else other_logp
        m64 = 2 ** 64 - 1
        if use_tc:
            # tensor-core path: both networks' row tiles share one persistent grid (any batch size)
            if obs is None:
                obs, env, obs_stats, obs_out = self._tc_obs(env, obs_stats, obs_out), None, None, None
            L.check(self.lib.sat_actor_sample_pair_tc(C.byref(self.w), C.byref(other.w), self._image().data_ptr(),
                                                      other._image().data_ptr(), L.ptr(obs),
                                                      C.byref(env.st) if env is not None else None,
                                                      L.ptr(obs_stats.buf) if obs_stats is not None else None, n,
                                                      int(row_offset), int(seed) & m64, int(step) & m64, int(other_step) & m64,
                                                      L.ptr(act), L.ptr(logp), L.ptr(obs_out), L.ptr(other_act),
                                                      L.ptr(other_logp), L.stream_ptr()), "sat_actor_sample_pair_tc")
            return act, logp, other_act, other_logp
        L.check(self.lib.sat_actor_sample_pair(C.byref(self.w), C.byref(other.w), L.ptr(obs),
                                               C.byref(env.st) if env is not None else None,
                                               L.ptr(obs_stats.buf) if obs_stats is not None else None, n, int(row_offset),
                                               int(seed) & m64, int(step) & m64, int(other_step) & m64, L.ptr(act), L.ptr(logp),
                                               L.ptr(obs_out), L.ptr(other_act), L.ptr(other_logp), L.stream_ptr()),
                "sat_actor_sample_pair")
        return act, logp, other_act, other_logp

    def sample_vs_pool(self, pool: "OpponentPool", slots, group_row_end, obs=None, env: EnvBatch | None = None,
                       obs_stats: RunningStats | None = None, seed: int = 0, step: int = 0, other_step: int = 1,
                       row_offset: int = 0, act=None, logp=None, obs_out=None, other_act=None, other_logp=None,
                       tc: bool | None = None):
        """the pool counterpart of sample_pair: this actor on all rows (exactly sample_pair's own outputs) and, on rows
        [group_row_end[k - 1], group_row_end[k]), the snapshot in pool slot slots[k] (exactly that snapshot's sample() on
        those rows with row_offset + group_row_end[k - 1] and step other_step) -> (act, logp, other_act, other_logp).
        Tensor-core path (default): every group's tiles and the learner's go through ONE persistent grid
        (sat_actor_sample_pool_tc); every bound but the last a multiple of 128, the last = the row count. FFMA2 path
        (tc=False): one sample() per group."""
        torch = self.torch
        L.guard_device(self.device)
        if self.w is None:
            raise L.SatError("weights not loaded")
        slots, ends = [int(s) for s in slots], [int(e) for e in group_row_end]
        if len(slots) != len(ends):
            raise L.SatError(f"{len(slots)} slots for {len(ends)} groups")
        groups = [pool.group(s) for s in slots]                    # IndexError on a slot the pool does not hold
        n = obs.shape[0] if obs is not None else env.n
        use_tc = (self.use_tc if tc is None else tc) and not self.critic
        new = lambda: torch.empty((n, ACT_DIM), dtype=torch.float32, device=self.device)
        act = new() if act is None else act
        logp = new() if logp is None else logp
        other_act = new() if other_act is None else other_act
        other_logp = new() if other_logp is None else other_logp
        if obs is None:
            # the fp32 (normalised) observation, materialised once (sat_env_observe_norm: the fused path's arithmetic)
            obs, env, obs_stats, obs_out = self._tc_obs(env, obs_stats, obs_out), None, None, None
        m64 = 2 ** 64 - 1
        if use_tc:
            arr = (L.SatActorPoolGroup * max(1, len(groups)))()
            for k, (g, e) in enumerate(zip(groups, ends)):
                arr[k] = g
                arr[k].row_end = e
            L.check(self.lib.sat_actor_sample_pool_tc(C.byref(self.w), self._image().data_ptr(), arr, len(groups), L.ptr(obs),
                                                      None, None, n, int(row_offset), int(seed) & m64, int(step) & m64,
                                                      int(other_step) & m64, L.ptr(act), L.ptr(logp), L.ptr(obs_out),
                                                      L.ptr(other_act), L.ptr(other_logp), L.stream_ptr()),
                    "sat_actor_sample_pool_tc")
            return act, logp, other_act, other_logp
        if not 1 <= len(ends) <= L.ACTOR_POOL_MAX_GROUPS:
            raise L.SatError(f"{len(ends)} groups: 1 .. {L.ACTOR_POOL_MAX_GROUPS} supported")
        lo = 0
        for k, e in enumerate(ends):
            if e <= lo or (k + 1 < len(ends) and e % 128) or (k + 1 == len(ends) and e != n):
                raise L.SatError(f"group bounds {ends}: strictly increasing, multiples of 128 but the last, the last = {n}")
            lo = e
        if any(g.use_tanh != self.use_tanh for g in groups):
            raise L.SatError("a snapshot was built with another activation than this actor")
        self.sample(obs=obs, seed=seed, step=step, row_offset=row_offset, act=act, logp=logp, obs_out=obs_out, tc=False)
        lo = 0
        for s, e in zip(slots, ends):
            pool.kernel(s).sample(obs=obs[lo:e], seed=seed, step=other_step, row_offset=int(row_offset) + lo,
                                  act=other_act[lo:e], logp=other_logp[lo:e], tc=False)
            lo = e
        return act, logp, other_act, other_logp

    def value(self, obs, out=None):
        torch = self.torch
        if not self.critic:
            raise L.SatError("not a critic kernel")
        n = obs.shape[0]
        out = torch.empty(n, dtype=torch.float32, device=self.device) if out is None else out
        L.check(self.lib.sat_critic_forward(C.byref(self.w), L.ptr(obs), n, L.ptr(out), L.stream_ptr()),
                "sat_critic_forward")
        return out


class OpponentPool:
    """A FIFO ring of up to `capacity` frozen snapshots of an actor, for self-play against past opponents (fictitious
    self-play / league training instead of pure alternating best response). add(actor_kernel) copies the actor's packed
    weights and builds their tensor-core weight image and bias / head tables once (sat_actor_tc_snapshot, about 0.8 MB of
    device memory per snapshot); when the ring is full the oldest snapshot goes. Every snapshot gets the next id of a
    counter that never goes back. Slot k is the k-th oldest snapshot held (ids[k]). GaussianActorKernel.sample_vs_pool
    samples any of them on groups of rows in the learner's launch."""

    def __init__(self, capacity: int, use_tanh: bool = True, max_action: float = 1.6, device="cuda"):
        if not 1 <= int(capacity) <= L.ACTOR_POOL_MAX_GROUPS:
            raise L.SatError(f"pool capacity {capacity}: 1 .. {L.ACTOR_POOL_MAX_GROUPS} supported")
        torch = L.require_cuda()
        self.torch, self.lib = torch, L.load()
        self.capacity, self.use_tanh, self.max_action = int(capacity), int(bool(use_tanh)), float(max_action)
        self.device = torch.device(device)
        self._snaps = []                  # oldest first: {"id", "packed", "image", "tables", "group", "kernel"}
        self._next_id = 0

    def __len__(self):
        return len(self._snaps)

    @property
    def ids(self):
        return [s["id"] for s in self._snaps]

    def add(self, actor_kernel: GaussianActorKernel) -> int:
        """snapshot the actor's current weights; returns the snapshot's id"""
        if actor_kernel.w is None or actor_kernel.critic:
            raise L.SatError("the pool takes loaded actor kernels")
        if actor_kernel.use_tanh != self.use_tanh or actor_kernel.max_action != self.max_action:
            raise L.SatError("the actor's activation / max_action differ from the pool's")
        L.guard_device(self.device)
        s = self._snaps.pop(0) if len(self._snaps) == self.capacity else self._alloc()
        s["packed"].copy_(actor_kernel.packed)
        self._build(s)
        s["id"] = self._next_id
        self._next_id += 1
        self._snaps.append(s)
        return s["id"]

    def _alloc(self):
        torch = self.torch
        f32 = dict(dtype=torch.float32, device=self.device)
        s = {"packed": torch.empty(L.ACTOR_PACKED_FLOATS, **f32), "image": torch.empty(L.ACTOR_TC_IMAGE_FLOATS, **f32),
             "tables": torch.empty(L.ACTOR_TC_TABLE_FLOATS, **f32)}
        # the snapshot as a GaussianActorKernel (FFMA2 path and references): its own image scratch, so sample(tc=True)
        # never writes into the frozen image
        k = GaussianActorKernel(self.max_action, bool(self.use_tanh), self.device)
        k.packed = s["packed"]
        k.w = L.SatActorWeights(None, None, None, None, None, None, None, s["packed"].data_ptr(), OBS_DIM, 256, ACT_DIM,
                                self.use_tanh, self.max_action)
        s["kernel"] = k
        return s

    def _build(self, s):
        g = L.SatActorPoolGroup()
        L.check(self.lib.sat_actor_tc_snapshot(C.byref(s["kernel"].w), s["image"].data_ptr(), s["tables"].data_ptr(),
                                               C.byref(g), L.stream_ptr()), "sat_actor_tc_snapshot")
        s["group"] = g

    def group(self, slot: int):
        """the SatActorPoolGroup of slot `slot` (row_end 0)"""
        return self._snaps[slot]["group"]

    def kernel(self, slot: int) -> GaussianActorKernel:
        """the snapshot in slot `slot` as an actor kernel (do not train it)"""
        return self._snaps[slot]["kernel"]

    def state_dict(self):
        """packed weights and ids; the images and tables are rebuilt on load"""
        return {"capacity": self.capacity, "use_tanh": self.use_tanh, "max_action": self.max_action,
                "next_id": self._next_id, "ids": self.ids, "packed": [s["packed"].clone() for s in self._snaps]}

    def load_state_dict(self, sd):
        if int(sd["use_tanh"]) != self.use_tanh or float(sd["max_action"]) != self.max_action:
            raise L.SatError("the saved pool's activation / max_action differ from this pool's")
        if len(sd["packed"]) > self.capacity:
            raise L.SatError(f"the saved pool holds {len(sd['packed'])} snapshots, more than this pool's capacity {self.capacity}")
        L.guard_device(self.device)
        snaps = self._snaps
        self._snaps = []
        for i, (sid, packed) in enumerate(zip(sd["ids"], sd["packed"])):
            s = snaps[i] if i < len(snaps) else self._alloc()
            s["packed"].copy_(packed)
            self._build(s)
            s["id"] = int(sid)
            self._snaps.append(s)
        self._next_id = int(sd["next_id"])
        return self


# --------------------------------------------------------------------------------------------- fused PPO step
class PpoFusedNet:
    """One network of the fused PPO minibatch step (csrc/ppo_update.cu): flat parameter / gradient / Adam-moment buffers in
    torch parameter order. `adopt(module)` re-points the torch parameters at views of the flat buffer, so the module, its
    checkpoints and the eager PyTorch path keep seeing the weights this class updates."""

    ACTOR_NAMES = ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "mean_layer.weight", "mean_layer.bias", "log_std")
    CRITIC_NAMES = ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias")

    def __init__(self, module, critic: bool, use_tanh: bool, max_action: float, lr, packed=None, betas=(0.9, 0.999),
                 eps: float = 1e-8):
        torch = L.require_cuda()
        self.torch, self.lib, self.module, self.critic = torch, L.load(), module, critic
        self.heads = 1 if critic else 3
        self.n = L.ppo_param_floats(self.heads)
        dev = next(module.parameters()).device
        self.device = dev
        self.params = torch.zeros(self.n + 2, dtype=torch.float32, device=dev)
        # [n] = minibatch loss, [n + 2, n + 6) = the actor's diagnostics (stats variant); `grads` is the first n + 2 floats,
        # what the gradient exchange carries with stats off, `grads_stats` the whole buffer
        self.n_stats = L.ppo_grad_floats_stats(self.heads)
        self._own_grads = torch.zeros(self.n_stats, dtype=torch.float32, device=dev)
        self._set_grads(self._own_grads)
        self.exp_avg = torch.zeros(self.n + 2, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(self.n + 2, dtype=torch.float32, device=dev)
        self.step = torch.zeros(1, dtype=torch.int64, device=dev)
        self.packed = packed if packed is not None else torch.zeros(L.ACTOR_PACKED_FLOATS, dtype=torch.float32, device=dev)
        self.lr = lr                                                                 # fp32 device scalar, shared with torch's Adam
        self.betas, self.eps = betas, float(eps)
        self.use_tanh, self.max_action = int(bool(use_tanh)), float(max_action)
        self.workspace = None
        self.net = None
        self._peer = None
        self.adopt()

    # ---- multi-GPU: gradient all-reduce fused into the Adam kernel over NVLink peer memory
    def enable_peer_allreduce(self, group=None):
        """Moves the flat gradient into a torch symmetric-memory allocation (two halves, alternated per step) that every
        rank of `group` maps; `adam()` then orders the ranks with the allocation's device-side barrier and the Adam kernel
        sums all ranks' gradients itself (sat_ppo_adam_peers) - no NCCL call on the step."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        torch = self.torch
        g = group if group is not None else dist.group.WORLD
        stride = _round_up(self.n_stats, 64)
        buf = symm.empty(2 * stride, dtype=torch.float32, device=self.device)
        hdl = symm.rendezvous(buf, g.group_name)
        buf.zero_()
        self._peer = {"buf": buf, "hdl": hdl, "stride": stride, "parity": 0, "world": int(hdl.world_size),
                      "ptrs": int(hdl.buffer_ptrs_dev)}
        self._set_grads(buf[:self.n_stats])
        hdl.barrier()
        return self

    def disable_peer_allreduce(self):
        """back to a private gradient buffer (used when the symmetric-memory rendezvous did not succeed on EVERY rank)"""
        if self._peer is not None or self.grads.data_ptr() != self._own_grads.data_ptr():
            self._peer = None
            self._set_grads(self._own_grads)
        return self

    def _set_grads(self, buf):
        self.grads_stats = buf
        self.grads = buf[:self.n + 2]
        if getattr(self, "net", None) is not None:
            self.net.grads = self.grads.data_ptr()

    def _slices(self):
        names = self.CRITIC_NAMES if self.critic else self.ACTOR_NAMES
        named = dict(self.module.named_parameters())
        off = 0
        for k in names:
            p = named[k]
            yield p, off
            off += p.numel()
        if off != self.n:
            raise L.SatError(f"unexpected parameter count {off} (the fused step is built for 18-256-256-{self.heads})")

    def adopt(self):
        torch = self.torch
        with torch.no_grad():
            for p, off in self._slices():
                view = self.params[off:off + p.numel()].view(p.shape)
                if p.data_ptr() != view.data_ptr():
                    view.copy_(p.data)
                    p.data = view
        self.pack()

    def adopted(self) -> bool:
        return all(p.data_ptr() == self.params.data_ptr() + 4 * off for p, off in self._slices())

    def bind(self, workspace):
        self.workspace = workspace
        self.net = L.SatPpoNet(self.params.data_ptr(), self.packed.data_ptr(), self.grads.data_ptr(), self.exp_avg.data_ptr(),
                               self.exp_avg_sq.data_ptr(), workspace.data_ptr(), self.heads, self.use_tanh, self.max_action, 0)

    def pack(self):
        if self.net is None:
            self.bind(self.torch.zeros(4, dtype=self.torch.float32, device=self.device) if self.workspace is None else self.workspace)
        L.check(self.lib.sat_ppo_pack(C.byref(self.net), L.stream_ptr()), "sat_ppo_pack")

    def actor_weights(self):
        """SatActorWeights over the flat buffer (for sat_actor_sample / sat_critic_forward)."""
        b = self.params.data_ptr()
        o3 = L.PPO_OFF_W3
        return L.SatActorWeights(b + 4 * L.PPO_OFF_W1, b + 4 * L.PPO_OFF_B1, b + 4 * L.PPO_OFF_W2, b + 4 * L.PPO_OFF_B2,
                                 b + 4 * o3, b + 4 * (o3 + 256 * self.heads),
                                 None if self.critic else b + 4 * (o3 + 257 * self.heads), self.packed.data_ptr(),
                                 18, 256, self.heads, self.use_tanh, self.max_action)

    def actor_grad(self, s, a, old_logp, adv, index, mb, epsilon, entropy_coef, stats=False):
        """stats: also the minibatch's diagnostics in grads_stats[n + 2:] (sat_ppo_actor_grad_stats; same gradient bits)"""
        fn, name = (self.lib.sat_ppo_actor_grad_stats, "sat_ppo_actor_grad_stats") if stats else (self.lib.sat_ppo_actor_grad, "sat_ppo_actor_grad")
        L.check(fn(C.byref(self.net), L.ptr(s), L.ptr(a), L.ptr(old_logp), L.ptr(adv), index, mb, float(epsilon),
                   float(entropy_coef), L.stream_ptr()), name)

    def critic_grad(self, s, v_target, index, mb):
        L.check(self.lib.sat_ppo_critic_grad(C.byref(self.net), L.ptr(s), L.ptr(v_target), index, mb, L.stream_ptr()),
                "sat_ppo_critic_grad")

    def adam(self, max_grad_norm: float, grad_scale: float = 1.0, record=None):
        """record: fp64 device tensor [PPO_STATS_DOUBLES] the step adds this minibatch's global statistics to
        (sat_ppo_adam_stats; same parameter bits)"""
        pr = self._peer
        args = (C.byref(self.net), L.ptr(self.lr), self.betas[0], self.betas[1], self.eps, float(max_grad_norm),
                float(grad_scale), L.ptr(self.step))
        if record is not None and (record.dtype != self.torch.float64 or record.numel() != L.PPO_STATS_DOUBLES):
            raise L.SatError(f"record must be {L.PPO_STATS_DOUBLES} fp64 values")
        if pr is None:
            if record is None:
                L.check(self.lib.sat_ppo_adam(*args, L.stream_ptr()), "sat_ppo_adam")
            else:
                L.check(self.lib.sat_ppo_adam_stats(*args, L.ptr(record), L.stream_ptr()), "sat_ppo_adam_stats")
            return
        # every rank's gradient kernels for this step are stream-ordered before its barrier; a rank can run at most one
        # step ahead of the slowest (the next barrier holds it), hence the two alternating halves of the buffer
        pr["hdl"].barrier()
        off = pr["parity"] * pr["stride"]
        if record is None:
            L.check(self.lib.sat_ppo_adam_peers(*args, pr["ptrs"], pr["world"], off, L.stream_ptr()), "sat_ppo_adam_peers")
        else:
            L.check(self.lib.sat_ppo_adam_peers_stats(*args, pr["ptrs"], pr["world"], off, L.ptr(record), L.stream_ptr()),
                    "sat_ppo_adam_peers_stats")
        pr["parity"] ^= 1
        off = pr["parity"] * pr["stride"]
        self._set_grads(pr["buf"][off:off + self.n_stats])

    def state_dict(self):
        return {"exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(), "step": self.step.clone()}

    def load_state_dict(self, sd):
        self.exp_avg.copy_(sd["exp_avg"]); self.exp_avg_sq.copy_(sd["exp_avg_sq"]); self.step.copy_(sd["step"])


def ppo_workspace(mb: int, device):
    torch = L.require_cuda()
    return torch.empty(int(L.load().sat_ppo_workspace_floats(int(mb))), dtype=torch.float32, device=device)


# --------------------------------------------------------------------------------------------- K4
def gae_time_major(r, v, done, gamma=0.99, lamda=0.95, r_scale=None, adv=None, v_target=None):
    """r [T,N] fp32, v [T+1,N] fp32, done [T,N] uint8 (CUDA). ppo_continuous.py:198-208 per env column."""
    torch = L.require_cuda()
    T, N = r.shape
    adv = torch.empty_like(r) if adv is None else adv
    v_target = torch.empty_like(r) if v_target is None else v_target
    L.check(L.load().sat_gae(L.ptr(r), L.ptr(v), L.ptr(done), L.ptr(r_scale), T, N, float(gamma), float(lamda),
                             L.ptr(adv), L.ptr(v_target), L.stream_ptr()), "sat_gae")
    return adv, v_target


def gae_flat(r, vs, vs_next, dw, done, gamma=0.99, lamda=0.95):
    """The reference's (B,1) buffers of one env in time order (all CUDA fp32)."""
    torch = L.require_cuda()
    r, vs, vs_next, dw, done = (t.reshape(-1).contiguous() for t in (r, vs, vs_next, dw, done))
    adv = torch.empty_like(r)
    vt = torch.empty_like(r)
    L.check(L.load().sat_gae_flat(L.ptr(r), L.ptr(vs), L.ptr(vs_next), L.ptr(dw), L.ptr(done), r.numel(),
                                  float(gamma), float(lamda), L.ptr(adv), L.ptr(vt), L.stream_ptr()), "sat_gae_flat")
    return adv, vt


def adv_moments(adv):
    """(sum, sum of squares, count) of a CUDA fp32 tensor as a 3-element fp64 CUDA tensor."""
    torch = L.require_cuda()
    sums = torch.empty(3, dtype=torch.float64, device=adv.device)
    ws = torch.empty(4096 * 2, dtype=torch.float64, device=adv.device)
    L.check(L.load().sat_adv_moments(L.ptr(adv.reshape(-1)), adv.numel(), L.ptr(sums), L.ptr(ws), L.stream_ptr()),
            "sat_adv_moments")
    return sums


def adv_normalize_(adv, sums=None, group=None):
    """in-place (adv-mean)/(std_unbiased+1e-5) (ppo_continuous.py:210); with `group` the three moments are
    all-reduced across ranks first, so every rank normalises with the global statistics."""
    torch = L.require_cuda()
    if sums is None:
        sums = adv_moments(adv)
    dist = torch.distributed
    if group is not False and dist.is_available() and dist.is_initialized():
        pg = None if group in (None, True) else group
        if dist.get_world_size(pg) > 1:
            dist.all_reduce(sums, group=pg)
    flat = adv.reshape(-1)
    L.check(L.load().sat_adv_normalize(L.ptr(flat), flat.numel(), L.ptr(sums), L.stream_ptr()), "sat_adv_normalize")
    return adv


# --------------------------------------------------------------------------------------------- peaks
def measure_vector_peak(dtype="fp64", iters=4096, repeats=5):
    """TFLOP/s of a dependent-free FMA chain kernel on the current device (roofline denominator)."""
    torch = L.require_cuda()
    lib = L.load()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    blocks, threads = sms * 8, 256
    flops = C.c_double()
    if dtype == "fp64":
        sink = torch.zeros(1, dtype=torch.float64, device="cuda")
        fn = lib.sat_peak_fp64
    else:
        sink = torch.zeros(1, dtype=torch.float32, device="cuda")
        fn = lib.sat_peak_fp32
        if dtype == "fp32x2":          # packed FFMA2 chains (negative iters selects them)
            iters = -iters
    best = 0.0
    for i in range(repeats + 2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(fn(sink.data_ptr(), blocks, threads, iters, C.byref(flops), L.stream_ptr()), "sat_peak")
        e1.record()
        e1.synchronize()
        if i >= 2:
            best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best
