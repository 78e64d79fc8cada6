"""Host-side mirror of the reference's MPC agent interface, backed by libmpcb200.so.

Reference surface reproduced (file:line in SaeedRahmani/MPC-RL_for_AVs):
  * `MPC_Action`                       agents/utils.py:4-12
  * `PureMPC_Agent(env, cfg)`          agents/pure_mpc.py:24-63, agents/base_agent.py:14-49
  * `PureMPC_Agent.predict(obs, return_numpy=True, weights_from_RL=None, ref_speed=None)`
                                       agents/pure_mpc.py:68-78
  * errors of `_parse_obs`             agents/base_agent.py:88-91
  * the no-collision variant           agents/pure_mpc_no_collision.py:12-64

plus the batched entry point the reference lacks (it solves one env at a time,
agents/a2c_mpc.py:145-150): `BatchedPureMPC.predict_batch`.

PyTorch is the batch container (device memory, streams); every number is produced by the CUDA
kernels.  Nothing here computes on the CPU and nothing falls back.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional, Union

import numpy as np
import torch

from . import _capi
from .scenarios import reference_path


class MPC_Action:
    """Result type of the reference agent (agents/utils.py:4-12)."""

    def __init__(self, acceleration, steer) -> None:
        self.acceleration = acceleration
        self.steer = steer

    def numpy(self) -> np.ndarray:
        return np.array([self.acceleration, self.steer])


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class BatchedPureMPC:
    """Thousands of independent PureMPC problems per call on one B200.

    cfg keys follow config/cfg.yaml:88-106 (`horizon`, `weight_speed`, `weight_control`,
    `weight_input_diff`).  The YAML's `weight_distance` / `weight_collision` are NOT read from cfg:
    the live agent's objective omits both terms (agents/pure_mpc.py:82, 204-212), so they are
    explicit constructor arguments defaulting to 0; pass `weight_distance=cfg["weight_distance"]`
    for the archive objective (agents/archive/pure_mpc.py:189-226, BASELINE config 3).

    n_starts: the NLP is multi-modal, so every problem is solved from `n_starts` starts (0 = the library default, 4)
    and the lowest objective wins; start 0 is the reference's own cold start (zero controls,
    agents/pure_mpc.py:244) and `n_starts=1` solves only that one (about 2.5x the throughput); `n_starts=2` adds the
    path-following start that finds the best optimum most often (DESIGN.md 2).

    `set_adaptive_starts(max_starts, rel_gap)` (opt-in) runs starts n_starts..max_starts-1 only for the problems whose
    first n_starts objectives disagree: most of the J_gpu <= J_oracle gain of max_starts starts for a fraction of their
    solves.  It trades a longer launch tail (a problem whose last base start ends late adds its extra solves at the end)
    for the solves skipped on problems where the base starts agree; each problem's result is bit-identical to a fixed
    portfolio of n_starts or max_starts starts."""

    def __init__(self, cfg: Dict, vehicles_count: int, max_batch: int, device: Union[int, str, torch.device] = 0,
                 dt: float = 0.1, collision_check: bool = True, literal_no_collision: bool = False,
                 weight_distance: float = 0.0, weight_collision: float = 0.0,
                 max_iter: int = 60, tol_step: float = 1e-4, reg_min: float = 1e-2,
                 threads_per_block: int = 0, blocks_per_sm: int = 0, n_starts: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("BatchedPureMPC needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("BatchedPureMPC needs a CUDA device (B200, sm_100a); there is no CPU path")
        self._lib = _capi.load()
        self.horizon = int(cfg["horizon"])
        self.vehicles_count = int(vehicles_count)
        self.n_obstacles = self.vehicles_count - 1
        self.max_batch = int(max_batch)
        self.dt = float(dt)
        self.collision_check = bool(collision_check)
        self.n_starts = int(n_starts) if int(n_starts) > 0 else 4
        c = _capi.MpcConfig(
            abi_version=_capi.ABI_VERSION, horizon=self.horizon, vehicles_count=self.vehicles_count, dt=self.dt,
            weight_speed=float(cfg.get("weight_speed", 1.0)), weight_control=float(cfg.get("weight_control", 1.0)),
            weight_input_diff=float(cfg.get("weight_input_diff", 1.0)),
            weight_distance=float(weight_distance), weight_collision=float(weight_collision),
            collision_check=int(collision_check), literal_no_collision=int(literal_no_collision),
            max_iter=int(max_iter), tol_step=float(tol_step), reg_min=float(reg_min),
            threads_per_block=int(threads_per_block), blocks_per_sm=int(blocks_per_sm), n_starts=int(n_starts))
        self._cfg = c
        h = C.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        rc = self._lib.mpc_create(C.byref(c), idx, self.max_batch, C.byref(h))
        _capi.check(self._lib, None, rc)
        self._h = h
        self.device = torch.device("cuda", idx)
        B, M = self.max_batch, max(self.n_obstacles, 1)
        dev = self.device
        # per-environment latch (agents/pure_mpc.py:38-43) -- caller-visible, resettable
        self.collision_memory = torch.zeros(B, dtype=torch.int32, device=dev)
        self.memo_conflict = torch.full((B,), -1, dtype=torch.int32, device=dev)
        self.latch_is_collide = torch.zeros(B, dtype=torch.uint8, device=dev)
        # outputs (public attributes of the reference agent, tensor-valued)
        self.actions = torch.zeros(B, 2, dtype=torch.float32, device=dev)
        self.status = torch.zeros(B, dtype=torch.int32, device=dev)
        self.iters = torch.zeros(B, dtype=torch.int32, device=dev)
        self.cost = torch.zeros(B, dtype=torch.float32, device=dev)
        self.is_collide = torch.zeros(B, dtype=torch.uint8, device=dev)
        self.agent_collide = torch.zeros(B, M, dtype=torch.uint8, device=dev)
        self.conflict_index = torch.full((B, M), -1, dtype=torch.int32, device=dev)
        self.ego_index = torch.zeros(B, dtype=torch.int32, device=dev)
        self.stop_index = torch.full((B,), -1, dtype=torch.int32, device=dev)
        self.degenerate = torch.zeros(B, dtype=torch.uint8, device=dev)
        self.conflict_point = torch.full((B, M, 2), float("nan"), dtype=torch.float32, device=dev)
        self.reference_trajectory = torch.from_numpy(reference_path(self.dt)[:, :2].copy()).to(dev)
        self._u_init = None
        self.max_starts = 0
        self.start_cost = None
        self.extended = None

    # ------------------------------------------------------------------ lifecycle
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.mpc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, mask: Optional[torch.Tensor] = None) -> None:
        """Clear the collision latch of the flagged environments (all if mask is None).  The
        reference never resets it (SURVEY quirk Q7); a vectorised caller needs to on `done`."""
        if mask is None:
            self.collision_memory.zero_(); self.memo_conflict.fill_(-1); self.latch_is_collide.zero_()
        else:
            m = mask.to(self.device).bool()
            n = m.shape[0]
            self.collision_memory[:n][m] = 0
            self.memo_conflict[:n][m] = -1
            self.latch_is_collide[:n][m] = 0

    def bind_actions(self, actions: Optional[torch.Tensor]) -> None:
        """Redirects the solver's action output to a caller-owned [>= max_batch, 2] float32 buffer on this
        device (e.g. this rank's slice of `sharding.ActionGather.buffer`, so the collective needs no copy).
        None restores the agent's own buffer."""
        if actions is None:
            self.actions = torch.zeros(self.max_batch, 2, dtype=torch.float32, device=self.device)
            return
        if (actions.device != self.device or actions.dtype != torch.float32 or not actions.is_contiguous()
                or actions.dim() != 2 or actions.shape[1] != 2):
            raise ValueError("actions must be a contiguous float32 [n, 2] tensor on this agent's CUDA device")
        self.actions = actions

    # ------------------------------------------------------------------ helpers
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check_obs(self, obs: torch.Tensor) -> int:
        if not isinstance(obs, torch.Tensor):
            raise TypeError(f"Expect observation type torch.Tensor, but got {type(obs)}.")
        if obs.dim() != 3 or tuple(obs.shape[1:]) != (self.vehicles_count, 8):
            raise ValueError(f"Expect observation's shape of (B, {self.vehicles_count}, 8), but got {tuple(obs.shape)}")
        if obs.shape[0] > self.max_batch or obs.shape[0] > self.actions.shape[0]:
            raise ValueError(f"batch {obs.shape[0]} exceeds max_batch {self.max_batch} / the bound action buffer")
        if obs.device != self.device or obs.dtype != torch.float32 or not obs.is_contiguous():
            raise ValueError("obs must be a contiguous float32 tensor on this agent's CUDA device")
        return int(obs.shape[0])

    def _norm_ref_speed(self, ref_speed, B):
        if ref_speed is None:
            return None
        r = ref_speed.to(device=self.device, dtype=torch.float32).reshape(-1).contiguous()
        if r.numel() != B:
            raise ValueError(f"ref_speed must have {B} entries, got {r.numel()}")
        return r

    def _norm_weights(self, weights, B):
        if weights is None:
            return None
        w = weights.to(device=self.device, dtype=torch.float32).reshape(B, -1)[:, :3].contiguous()
        if w.shape[1] != 3:
            raise ValueError("weights must have 3 columns (speed, control, input_diff)")
        return w

    def _solve_out(self, B: int, want_U: bool):
        U = torch.empty(B, self.horizon, 2, dtype=torch.float32, device=self.device) if want_U else None
        out = _capi.MpcSolveOut(actions=self.actions.data_ptr(), status=self.status.data_ptr(),
                                iters=self.iters.data_ptr(), cost=self.cost.data_ptr(), U=_ptr(U))
        return out, U

    # ------------------------------------------------------------------ the reference's predict(), batched
    def set_warm_start(self, u_init: Optional[torch.Tensor]) -> None:
        """OPT-IN (SURVEY N3): start the next solves from `u_init` [B, N, 2] (e.g. the previous solution
        shifted by one stage) instead of the reference's zero controls (agents/pure_mpc.py:240-246).
        None restores the cold start.  Changes which local optimum is found -- keep off for parity."""
        if u_init is None:
            self._u_init = None
            _capi.check(self._lib, self._h, self._lib.mpc_set_warm_start(self._h, None))
            return
        u = u_init.to(device=self.device, dtype=torch.float32).contiguous()
        if u.dim() != 3 or tuple(u.shape[1:]) != (self.horizon, 2):
            raise ValueError(f"u_init must be [B, {self.horizon}, 2]")
        self._u_init = u
        _capi.check(self._lib, self._h, self._lib.mpc_set_warm_start(self._h, u.data_ptr()))

    def set_adaptive_starts(self, max_starts: Optional[int], rel_gap: float = 1e-3) -> None:
        """OPT-IN adaptive portfolio: the next solves run starts n_starts..max_starts-1 only for problems whose first
        n_starts objectives disagree (one not finite, or max - min > rel_gap * max(|min|, 1)); the others keep the
        n_starts result.  After a call of B problems, `self.start_cost[:, :B]` holds every start's objective (NaN where
        a start did not run) and `self.extended[:B]` marks the problems that ran the extra starts.  None or 0 switches
        the mode off.  Allocates: call it outside CUDA graph capture."""
        if max_starts is None or int(max_starts) == 0:
            _capi.check(self._lib, self._h, self._lib.mpc_set_adaptive_starts(self._h, 0, 0.0, None, None))
            self.max_starts, self.start_cost, self.extended = 0, None, None
            return
        S = int(max_starts)
        if self.n_starts < 2:
            raise ValueError("the adaptive portfolio needs n_starts >= 2")
        if not self.n_starts < S <= _capi.MAX_STARTS:
            raise ValueError(f"max_starts must be in ({self.n_starts}, {_capi.MAX_STARTS}], got {S}")
        if math.isnan(float(rel_gap)):
            raise ValueError("rel_gap must not be NaN")
        if self.max_batch * S > 0x7FFFFFFF // 64:
            raise ValueError("max_batch * max_starts too large")
        start_cost = torch.full((S, self.max_batch), float("nan"), dtype=torch.float32, device=self.device)
        extended = torch.zeros(self.max_batch, dtype=torch.uint8, device=self.device)
        rc = self._lib.mpc_set_adaptive_starts(self._h, S, float(rel_gap), start_cost.data_ptr(), extended.data_ptr())
        _capi.check(self._lib, self._h, rc)
        self.max_starts, self.start_cost, self.extended = S, start_cost, extended

    @staticmethod
    def shift_controls(U: torch.Tensor) -> torch.Tensor:
        """Receding-horizon shift: u_k <- u_{k+1}, last stage repeated."""
        return torch.cat([U[:, 1:], U[:, -1:]], dim=1).contiguous()

    def predict_batch(self, obs: torch.Tensor, ref_speed: Optional[torch.Tensor] = None,
                      weights: Optional[torch.Tensor] = None, reset_mask: Optional[torch.Tensor] = None,
                      return_controls: bool = False):
        """obs [B,V,8] f32 cuda -> actions [B,2] f32 cuda (a view into `self.actions`).

        ref_speed [B,1] (NaN = no override) and weights [B,3] are the batched forms of
        `ref_speed` (1,1) / `weights_from_RL` (1,3) of agents/pure_mpc.py:68-78.  Runs on the
        current torch stream, no host synchronisation."""
        B = self._check_obs(obs)
        rs = self._norm_ref_speed(ref_speed, B)
        w = self._norm_weights(weights, B)
        rm = None if reset_mask is None else reset_mask.to(device=self.device, dtype=torch.uint8).contiguous()
        latch = _capi.MpcLatchState(self.collision_memory.data_ptr(), self.memo_conflict.data_ptr(),
                                    self.latch_is_collide.data_ptr())
        col = _capi.MpcCollisionOut(self.agent_collide.data_ptr(), self.conflict_index.data_ptr(),
                                    self.is_collide.data_ptr(), self.ego_index.data_ptr(), self.stop_index.data_ptr(),
                                    self.degenerate.data_ptr(), self.conflict_point.data_ptr())
        out, U = self._solve_out(B, return_controls)
        rc = self._lib.mpc_predict(self._h, obs.data_ptr(), _ptr(rs), _ptr(w), _ptr(rm), C.byref(latch), B,
                                   C.byref(out), C.byref(col), self._stream())
        _capi.check(self._lib, self._h, rc)
        self._keep = (obs, rs, w, rm)          # keep inputs alive until the stream has consumed them
        return (self.actions[:B], U) if return_controls else self.actions[:B]

    def prepare_batch(self, obs, ref_speed=None, weights=None, reset_mask=None) -> Dict[str, torch.Tensor]:
        """Parsing + collision logic only (mpc_prepare); returns the parsed-problem workspace as tensors
        (copies) for inspection / parity tests."""
        B = self._check_obs(obs)
        rs = self._norm_ref_speed(ref_speed, B)
        w = self._norm_weights(weights, B)
        rm = None if reset_mask is None else reset_mask.to(device=self.device, dtype=torch.uint8).contiguous()
        latch = _capi.MpcLatchState(self.collision_memory.data_ptr(), self.memo_conflict.data_ptr(),
                                    self.latch_is_collide.data_ptr())
        col = _capi.MpcCollisionOut(self.agent_collide.data_ptr(), self.conflict_index.data_ptr(),
                                    self.is_collide.data_ptr(), self.ego_index.data_ptr(), self.stop_index.data_ptr(),
                                    self.degenerate.data_ptr(), self.conflict_point.data_ptr())
        rc = self._lib.mpc_prepare(self._h, obs.data_ptr(), _ptr(rs), _ptr(w), _ptr(rm), C.byref(latch), B,
                                   C.byref(col), self._stream())
        _capi.check(self._lib, self._h, rc)
        self._keep = (obs, rs, w, rm)
        return self.workspace(B)

    def workspace(self, B: int) -> Dict[str, torch.Tensor]:
        """Copies of the handle's parsed-problem arrays (SoA, strided by max_batch) trimmed to B."""
        ws = _capi.MpcProblemBatch()
        _capi.check(self._lib, self._h, self._lib.mpc_workspace_batch(self._h, C.byref(ws)))
        torch.cuda.synchronize(self.device)
        MB, M = self.max_batch, max(self.n_obstacles, 1)

        def grab(ptr, n, dtype):
            class _Raw:      # device-pointer view through the CUDA array interface, then an owning copy
                pass
            r = _Raw()
            r.__cuda_array_interface__ = {"shape": (n,), "typestr": {torch.float32: "<f4", torch.int32: "<i4", torch.uint8: "|u1"}[dtype],
                                          "data": (int(ptr), False), "version": 2}
            with torch.cuda.device(self.device):
                return torch.as_tensor(r, device=self.device).clone()

        # mpc_prepare writes with stride B (the call's batch), not max_batch
        out = {
            "s0": grab(ws.s0, 4 * B, torch.float32).reshape(4, B),
            "ego_index": grab(ws.ego_index, B, torch.int32),
            "w_speed": grab(ws.w_speed, B, torch.float32),
            "w_control": grab(ws.w_control, B, torch.float32),
            "w_diff": grab(ws.w_diff, B, torch.float32),
            "vr_a": grab(ws.vr_a, B, torch.float32),
            "vr_slope": grab(ws.vr_slope, B, torch.float32),
            "vr_b": grab(ws.vr_b, B, torch.float32),
            "vr_n": grab(ws.vr_n, B, torch.int32),
            "is_collide": grab(ws.is_collide, B, torch.uint8),
            "n_obs": grab(ws.n_obs, B, torch.int32),
            "obstacles": grab(ws.obstacles, M * 4 * B, torch.float32).reshape(M, 4, B),
        }
        return out

    # ------------------------------------------------------------------ lower-level entry points
    def _batch_struct(self, batch: Dict[str, torch.Tensor]):
        need = ["s0", "ego_index", "w_speed", "w_control", "w_diff", "vr_a", "vr_slope", "vr_b", "vr_n"]
        for k in need:
            if k not in batch:
                raise ValueError(f"batch is missing '{k}'")
        B = int(batch["ego_index"].shape[0])
        dt = {"s0": torch.float32, "ego_index": torch.int32, "w_speed": torch.float32, "w_control": torch.float32,
              "w_diff": torch.float32, "vr_a": torch.float32, "vr_slope": torch.float32, "vr_b": torch.float32,
              "vr_n": torch.int32, "is_collide": torch.uint8, "n_obs": torch.int32, "obstacles": torch.float32}
        held = {}
        s = _capi.MpcProblemBatch()
        for k, d in dt.items():
            t = batch.get(k)
            if t is None:
                setattr(s, k, None)
                continue
            t = t.to(device=self.device, dtype=d).contiguous()
            held[k] = t
            setattr(s, k, t.data_ptr())
        if held["s0"].shape != (4, B):
            raise ValueError("s0 must be [4, B]")
        if "obstacles" in held and held["obstacles"].shape != (max(self.n_obstacles, 1), 4, B) and self.n_obstacles > 0:
            raise ValueError(f"obstacles must be [{self.n_obstacles}, 4, B]")
        return s, held, B

    def solve_batch(self, batch: Dict[str, torch.Tensor], return_controls: bool = False):
        """mpc_solve on caller-provided parsed problems (SoA tensors named as MpcProblemBatch)."""
        s, held, B = self._batch_struct(batch)
        if B > self.max_batch:
            raise ValueError("batch exceeds max_batch")
        out, U = self._solve_out(B, return_controls)
        rc = self._lib.mpc_solve(self._h, C.byref(s), B, C.byref(out), self._stream())
        _capi.check(self._lib, self._h, rc)
        self._keep = held
        return (self.actions[:B], U) if return_controls else self.actions[:B]

    def rollout_cost(self, batch: Dict[str, torch.Tensor], U: torch.Tensor):
        """K1 parity entry: X [B,N+1,4], cost6 [B,6] (state, control, final_state, input_diff, distance,
        collision -- the reference's cost_fn, agents/pure_mpc.py:215-216), total [B]."""
        s, held, B = self._batch_struct(batch)
        U = U.to(device=self.device, dtype=torch.float32).contiguous()
        if tuple(U.shape) != (B, self.horizon, 2):
            raise ValueError(f"U must be [B, {self.horizon}, 2]")
        X = torch.empty(B, self.horizon + 1, 4, dtype=torch.float32, device=self.device)
        c6 = torch.empty(B, 6, dtype=torch.float32, device=self.device)
        tot = torch.empty(B, dtype=torch.float32, device=self.device)
        rc = self._lib.mpc_rollout_cost(self._h, C.byref(s), B, U.data_ptr(), X.data_ptr(), c6.data_ptr(),
                                        tot.data_ptr(), self._stream())
        _capi.check(self._lib, self._h, rc)
        self._keep = (held, U)
        return X, c6, tot

    def predict_host(self, obs: np.ndarray, ref_speed: Optional[np.ndarray] = None,
                     weights: Optional[np.ndarray] = None, reset_mask: Optional[np.ndarray] = None,
                     collision_outputs: bool = False):
        """numpy in, numpy out (host<->device copies inside the call): the call a numpy-holding caller of
        the reference makes.  Uses the handle's own latch.  Returns (actions [B,2] f32, status [B] i32,
        is_collide [B] u8, h2d_bytes, d2h_bytes); with `collision_outputs` a sixth element: a dict with the per-call
        collision outputs (agent_collide [B,M], conflict_index [B,M], conflict_point [B,M,2], ego_index [B],
        stop_index [B], degenerate [B]) -- the public attributes of the reference agent."""
        if not isinstance(obs, np.ndarray):
            raise TypeError(f"Expect observation type np.ndarray, but got {type(obs)}.")
        if obs.ndim != 3 or obs.shape[1:] != (self.vehicles_count, 8):
            raise ValueError(f"Expect observation's shape of (B, {self.vehicles_count}, 8), but got {obs.shape}")
        B = obs.shape[0]
        if B > self.max_batch:
            raise ValueError(f"batch {B} exceeds max_batch {self.max_batch}")
        obs = np.ascontiguousarray(obs, dtype=np.float32)
        rs = None if ref_speed is None else np.ascontiguousarray(ref_speed, dtype=np.float32).reshape(-1)
        w = None if weights is None else np.ascontiguousarray(np.asarray(weights, dtype=np.float32).reshape(B, -1)[:, :3])
        rm = None if reset_mask is None else np.ascontiguousarray(reset_mask, dtype=np.uint8).reshape(-1)
        # the C side reads B entries of each: a shorter array would be read past its end
        if rs is not None and rs.size != B:
            raise ValueError(f"ref_speed must have {B} entries, got {rs.size}")
        if w is not None and w.shape != (B, 3):
            raise ValueError(f"weights must be [{B}, 3], got {w.shape}")
        if rm is not None and rm.size != B:
            raise ValueError(f"reset_mask must have {B} entries, got {rm.size}")
        actions = np.empty((B, 2), dtype=np.float32)
        status = np.empty(B, dtype=np.int32)
        iscol = np.empty(B, dtype=np.uint8)
        up, down = C.c_int64(0), C.c_int64(0)

        def p(a):
            return None if a is None else a.ctypes.data

        col, extra = None, None
        if collision_outputs:
            M = max(self.n_obstacles, 1)
            extra = dict(agent_collide=np.zeros((B, M), np.uint8), conflict_index=np.full((B, M), -1, np.int32),
                         ego_index=np.zeros(B, np.int32), stop_index=np.full(B, -1, np.int32), degenerate=np.zeros(B, np.uint8),
                         conflict_point=np.full((B, M, 2), np.nan, np.float32))
            col = _capi.MpcCollisionOut(p(extra["agent_collide"]), p(extra["conflict_index"]), None, p(extra["ego_index"]),
                                        p(extra["stop_index"]), p(extra["degenerate"]), p(extra["conflict_point"]))
        rc = self._lib.mpc_predict_host(self._h, p(obs), p(rs), p(w), p(rm), B, p(actions), p(status), p(iscol),
                                        None if col is None else C.byref(col), C.byref(up), C.byref(down))
        _capi.check(self._lib, self._h, rc)
        if collision_outputs:
            return actions, status, iscol, int(up.value), int(down.value), extra
        return actions, status, iscol, int(up.value), int(down.value)

    # ------------------------------------------------------------------ measurement hooks
    def launch_count(self) -> int:
        return int(self._lib.mpc_launch_count(self._h))

    def fp32_peak_tflops(self, repeats: int = 5) -> float:
        v = C.c_float(0)
        _capi.check(self._lib, self._h, self._lib.mpc_fp32_peak(self._h, repeats, C.byref(v)))
        return float(v.value)

    def timing_begin(self) -> None:
        _capi.check(self._lib, self._h, self._lib.mpc_timing_begin(self._h))

    def timing_end(self):
        a, b, na, nb = C.c_float(0), C.c_float(0), C.c_int(0), C.c_int(0)
        _capi.check(self._lib, self._h, self._lib.mpc_timing_end(self._h, C.byref(a), C.byref(b), C.byref(na), C.byref(nb)))
        return {"prepare_ms": float(a.value), "solve_ms": float(b.value), "n_prepare": na.value, "n_solve": nb.value}

    def solve_config(self, B: int):
        """Kernel and block size a launch of B problems uses (reporting only)."""
        a, b = C.c_int(0), C.c_int(0)
        _capi.check(self._lib, self._h, self._lib.mpc_solve_config(self._h, int(B), C.byref(a), C.byref(b)))
        return {"gains_in_tmem": bool(a.value), "threads_per_block": b.value}

    def device_info(self):
        a, b, c, d = C.c_int(0), C.c_int(0), C.c_int(0), C.c_int(0)
        _capi.check(self._lib, self._h, self._lib.mpc_device_info(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return {"sm_count": a.value, "cc": (b.value, c.value), "smem_optin": d.value}


class _EnvConfigView:
    """What the reference reads from `env.unwrapped.config` (agents/base_agent.py:28-34)."""

    def __init__(self, env):
        un = getattr(env, "unwrapped", env)
        cfg = un.config
        self.simulate_freq = int(cfg["simulation_frequency"])
        self.policy_freq = int(cfg["policy_frequency"])
        self.vehicles_count = int(cfg["observation"]["vehicles_count"])


class _VehicleView:
    """What callers and plots read from `agent.ego_vehicle` / `agent.agent_vehicles` (agents/utils.py:16-40)."""

    def __init__(self, index, row, heading):
        self.index = index
        self.is_ego = index == 0
        self.position = row[1:3]
        self.vectorized_speed = row[3:5]
        self.heading = heading
        self.speed = np.linalg.norm(self.vectorized_speed)
        self.sinh, self.cosh = row[6], row[7]
        self.max_acceleration = 3.5
        self.max_deceleration = -10


class PureMPC_Agent:
    """Drop-in for `agents.pure_mpc.PureMPC_Agent` (collision-aware) -- same constructor and
    `predict` signature, same return types, same two exceptions, same public attributes -- solving on the B200.

    `env` only needs `.unwrapped.config` (or `.config`) with `simulation_frequency`,
    `policy_frequency` and `observation.vehicles_count`.

    Attributes kept up to date by `predict` (read by the reference's scripts, plots and SB3 subclasses):
    `ego_index`, `is_collide`, `agent_collide`, `conflict_index`, `conflict_points`, `agent_current_locations`,
    `stop_point`, `last_valid_stop_point`, `collision_memory`, `last_acc`, `ego_vehicle`, `agent_vehicles`,
    `reference_trajectory`, `reference_states`.  `plot()` / `visualize_predictions()` exist and do nothing:
    matplotlib rendering is out of scope (`main/run_pure_mpc.py:32` calls `plot()` unconditionally)."""

    weight_components = ["speed", "control", "input_diff"]          # agents/pure_mpc.py:15-22
    _collision_check = True
    _literal = False

    def __init__(self, env, cfg: dict, device: Union[int, str] = 0, use_distance_cost: bool = False, n_starts: int = 0) -> None:
        ev = _EnvConfigView(env)
        self.env = getattr(env, "unwrapped", env)
        self.env_config = self.env.config
        self.config = cfg
        self.simulate_freq, self.policy_freq = ev.simulate_freq, ev.policy_freq
        self.total_vehicles_count = ev.vehicles_count
        self.horizon = cfg["horizon"]
        self.dt = 1 / self.policy_freq                               # agents/base_agent.py:43
        self.render = cfg.get("render", False)
        self.ttc_threshold = cfg.get("ttc_threshold", 3)
        self.default_weights = {f"weight_{k}": cfg[f"weight_{k}"] for k in PureMPC_Agent.weight_components}
        self.global_reference_states = reference_path(self.dt)
        self.reference_trajectory = self.global_reference_states[:, :2]
        self._solver = BatchedPureMPC(cfg, vehicles_count=self.total_vehicles_count, max_batch=1, device=device,
                                      dt=self.dt, collision_check=self._collision_check,
                                      literal_no_collision=self._literal, n_starts=n_starts,
                                      weight_distance=float(cfg.get("weight_distance", 0.0)) if use_distance_cost else 0.0)
        # per-instance state of agents/pure_mpc.py:38-43, :63 (the latch itself lives in the library handle)
        self.collision_memory = 0
        self.collision_memory_steps = 10
        self.memorized_conflict_points = None
        self.memorized_conflict_indices = None
        self.last_valid_stop_point = None
        self.stop_point = None
        self.last_acc = 0
        self.is_collide = False
        self.ego_index = 0
        self.status = 0
        self.agent_collide, self.conflict_index, self.conflict_points = [], [], []
        self.agent_current_locations, self.agent_vehicles, self.ego_vehicle = [], [], None
        self.observed_vehicles_count = 0

    def __str__(self) -> str:
        return "Pure MPC agent [Receding Horizon Control], solved by batched DDP on B200"

    @property
    def reference_states(self):
        return reference_path(self.dt)

    @staticmethod
    def normalize_angle(angle):
        """agents/base_agent.py:156-170."""
        while angle > np.pi:
            angle -= 2 * np.pi
        while angle < -np.pi:
            angle += 2 * np.pi
        return angle

    def plot(self, *args, **kwargs) -> None:
        """No-op: the matplotlib debug view of agents/pure_mpc.py:726-804 is out of scope."""

    def visualize_predictions(self, *args, **kwargs) -> None:
        """No-op: agents/pure_mpc.py:321-457 (matplotlib)."""

    def predict(self, obs, return_numpy=True, weights_from_RL=None, ref_speed=None):
        if not isinstance(obs, np.ndarray):
            raise TypeError(f"Expect observation type np.ndarray, but got {type(obs)}.")
        if obs.shape != (self.total_vehicles_count, 8):
            raise ValueError(f"Expect observation's shape of ({(self.total_vehicles_count, 8)}), but got {obs.shape}")
        rs = None if ref_speed is None else np.asarray(ref_speed, dtype=np.float32).reshape(-1)[:1]
        w = None if weights_from_RL is None else np.asarray(weights_from_RL, dtype=np.float32).reshape(1, -1)
        actions, status, iscol, _, _, col = self._solver.predict_host(obs[None], rs, w, collision_outputs=True)
        self.status = int(status[0])
        # what the reference prints when IPOPT reports failure (agents/pure_mpc.py:303-304); the iterate is applied
        # anyway, as there.  Settling on a kink of the clamped dynamics is not a failure; an infeasible s0 is one there too.
        if self.status & (_capi.STATUS_MAX_ITER | _capi.STATUS_LINESEARCH_FAIL | _capi.STATUS_NAN | _capi.STATUS_STALLED
                          | _capi.STATUS_INFEASIBLE_START):
            print("NOTICE: Not found solution")
        # ---- public attributes of the reference agent ----------------------------------------------------------------
        o = np.asarray(obs)
        n = max(int(np.sum(o[:, 0] == 1)) - 1, 0)
        n = min(n, self._solver.n_obstacles)
        self.observed_vehicles_count = n
        self.ego_vehicle = _VehicleView(0, o[0], self.normalize_angle(o[0, 5]))          # base_agent.py:95-102
        self.agent_vehicles = [_VehicleView(i + 1, o[i + 1], o[i + 1, 5]) for i in range(n)]
        self.ego_index = int(col["ego_index"][0])
        was_latched = self.collision_memory > 0 and self.memorized_conflict_points is not None
        self.is_collide = bool(iscol[0])
        if self._collision_check:
            if was_latched:                                        # pure_mpc.py:558-563: memorised values, no detection
                self.conflict_points = self.memorized_conflict_points
                self.conflict_index = self.memorized_conflict_indices
                self.collision_memory -= 1
            else:
                self.agent_current_locations = [v.position for v in self.agent_vehicles]
                self.agent_collide = [bool(x) for x in col["agent_collide"][0, :n]]
                self.conflict_index = [int(c) if f else None for c, f in zip(col["conflict_index"][0, :n], self.agent_collide)]
                self.conflict_points = [np.asarray(pt, dtype=np.float64) if f else None
                                        for pt, f in zip(col["conflict_point"][0, :n], self.agent_collide)]
                if self.is_collide and any(self.agent_collide):    # pure_mpc.py:664-668
                    self.collision_memory = self.collision_memory_steps
                    self.memorized_conflict_points = list(self.conflict_points)
                    self.memorized_conflict_indices = list(self.conflict_index)
                elif self.collision_memory > 0:
                    self.collision_memory -= 1
                else:
                    self.memorized_conflict_points = None
                    self.memorized_conflict_indices = None
            stop = int(col["stop_index"][0])
            if stop >= 0:                                          # pure_mpc.py:717-722
                self.stop_point = self.reference_trajectory[stop]
                self.last_valid_stop_point = self.stop_point
            elif self.is_collide and self.last_valid_stop_point is not None and ref_speed is None:
                self.stop_point = self.last_valid_stop_point
        a, d = float(actions[0, 0]), float(actions[0, 1])
        self.last_acc = a
        act = MPC_Action(acceleration=a, steer=d)
        return act.numpy() if return_numpy else act



class PureMPC_NoCollision_Agent(PureMPC_Agent):
    """Drop-in for `agents.pure_mpc_no_collision.PureMPC_Agent`: no collision check / regeneration.
    `literal=True` reproduces that file's objective exactly (state cost commented out,
    pure_mpc_no_collision.py:146-151 -- SURVEY quirk Q3); the default keeps the tracking objective."""

    _collision_check = False

    def __init__(self, env, cfg: dict, device: Union[int, str] = 0, literal: bool = False, n_starts: int = 0) -> None:
        self._literal = bool(literal)
        cfg = dict(cfg)
        cfg.setdefault("weight_speed", cfg.get("weight_state", 1.0) if literal else 1.0)   # quirk Q4
        super().__init__(env, cfg, device, n_starts=n_starts)
