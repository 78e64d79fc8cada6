"""Seeded synthetic intersection scenarios (SURVEY.md section 8-d).

Produces observations in highway-env's Kinematics layout consumed by the reference agent
(`config/config.py:13`: presence, x, y, vx, vy, heading, sin_h, cos_h; absolute, un-normalised),
float32, shape [B, V, 8] with row 0 the ego.  Geometry follows the intersection the reference
drives (`envs/intersection_env__.py:141-249`): lane centres at x = +-2 / y = +-2, the ego on
the hard-coded left-turn path of `agents/base_agent.py:118-154`.
"""
from __future__ import annotations

import math
from typing import Optional, Tuple

import numpy as np
import torch


def reference_path(dt: float = 0.1) -> np.ndarray:
    """(85, 4) rows (x, y, v, heading): the reference's hard-coded left-turn path
    (`agents/base_agent.py:118-154`), accumulated in the same order in FP64."""
    rows = []
    x, y, v, h = 2.0, 50.0, 10.0, -math.pi / 2
    for i in range(85):
        if i < 40:
            y += v * dt * math.sin(h)
        elif i < 60:
            h -= (math.pi / 2) / 20
            x += v * dt * math.cos(h)
            y += v * dt * math.sin(h)
        else:
            x += v * dt * math.cos(h)
        rows.append((x, y, v, h))
    return np.asarray(rows, dtype=np.float64)


_LANE_HEADING = np.array([-math.pi / 2, 0.0, math.pi / 2, math.pi])


def make_scenarios(batch: int, n_obstacles: int = 8, seed: int = 1234, vehicles_count: Optional[int] = None,
                   ref_speed_fraction: float = 0.5, v_max: float = 12.0, same_lane_frac: float = 0.0, dt: float = 0.1
                   ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Returns (obs [B,V,8] f32, ref_speed [B,1] f32, has_ref_speed [B] bool) on the CPU.

    Ego: reference row j ~ U{0..80}, lateral offset N(0, 0.3^2), longitudinal U(-0.5, 0.5),
    heading h_j + N(0, 0.05^2) wrapped to [-pi, pi], speed U(0, v_max).  Obstacles: approach
    c ~ U{0..3}, position R_c (2 + N(0, 0.2^2), d), d ~ U(-30, 70), speed max(0.5, N(8, 1)),
    lane heading; samples closer than 5 m to the ego are redrawn.  `ref_speed` ~ U(0, 15) for the
    flagged fraction of the batch (RL v0 mode), unused elsewhere.
    `same_lane_frac` > 0 (tests): in that fraction of the scenes the first other vehicle sits EXACTLY on the ego's lane
    centre x = 2.0 with heading -pi/2 (highway-env spawns on the lane centre, which is the reference path's own x) --
    the collinear / LineString branch of the reference's collision check (agents/pure_mpc.py:615-633).  Drawn from a
    separate stream so the default scenes do not change.
    `dt` (the policy step, 1 / policy_frequency): the ego is placed on `reference_path(dt)`, the path an agent with that
    policy frequency follows; the random draws do not depend on it.
    """
    g = torch.Generator(device="cpu")
    g.manual_seed(int(seed))
    V = vehicles_count if vehicles_count is not None else n_obstacles + 1
    if V < n_obstacles + 1:
        raise ValueError("vehicles_count must be >= n_obstacles + 1")
    ref = reference_path(dt)
    B, M = int(batch), int(n_obstacles)

    def randn(*s):
        return torch.randn(*s, generator=g, dtype=torch.float64).numpy()

    def rand(*s):
        return torch.rand(*s, generator=g, dtype=torch.float64).numpy()

    j = torch.randint(0, 81, (B,), generator=g).numpy()
    h = ref[j, 3]
    lat, lon = 0.3 * randn(B), rand(B) - 0.5
    ex = ref[j, 0] + lat * (-np.sin(h)) + lon * np.cos(h)
    ey = ref[j, 1] + lat * (np.cos(h)) + lon * np.sin(h)
    eth = h + 0.05 * randn(B)
    eth = np.where(eth > math.pi, eth - 2 * math.pi, eth)
    eth = np.where(eth < -math.pi, eth + 2 * math.pi, eth)
    ev = v_max * rand(B)

    obs = np.zeros((B, V, 8), dtype=np.float64)
    obs[:, 0, 0] = 1.0
    obs[:, 0, 1], obs[:, 0, 2] = ex, ey
    obs[:, 0, 3], obs[:, 0, 4] = ev * np.cos(eth), ev * np.sin(eth)
    obs[:, 0, 5], obs[:, 0, 6], obs[:, 0, 7] = eth, np.sin(eth), np.cos(eth)

    if M > 0:
        c = torch.randint(0, 4, (B, M), generator=g).numpy()
        lane = 2.0 + 0.2 * randn(B, M)
        d = -30.0 + 100.0 * rand(B, M)
        spd = np.maximum(0.5, 8.0 + randn(B, M))
        for _ in range(64):      # redraw the along-lane coordinate of samples too close to the ego
            ang = c * (math.pi / 2)
            px = np.cos(ang) * lane - np.sin(ang) * d
            py = np.sin(ang) * lane + np.cos(ang) * d
            close = np.hypot(px - ex[:, None], py - ey[:, None]) < 5.0
            if not close.any():
                break
            d = np.where(close, -30.0 + 100.0 * rand(B, M), d)
        hd = _LANE_HEADING[c]
        obs[:, 1:M + 1, 0] = 1.0
        obs[:, 1:M + 1, 1], obs[:, 1:M + 1, 2] = px, py
        obs[:, 1:M + 1, 3], obs[:, 1:M + 1, 4] = spd * np.cos(hd), spd * np.sin(hd)
        obs[:, 1:M + 1, 5], obs[:, 1:M + 1, 6], obs[:, 1:M + 1, 7] = hd, np.sin(hd), np.cos(hd)

    has = rand(B) < ref_speed_fraction
    rs = 15.0 * rand(B)
    if M > 0 and same_lane_frac > 0.0:
        g2 = torch.Generator(device="cpu")
        g2.manual_seed(int(seed) + 99991)
        pick = torch.rand(B, generator=g2, dtype=torch.float64).numpy() < same_lane_frac
        off = 6.0 + 30.0 * torch.rand(B, generator=g2, dtype=torch.float64).numpy()
        ahead = torch.rand(B, generator=g2, dtype=torch.float64).numpy() < 0.8
        y = np.where(ahead, ey - off, ey + off)              # ahead = further along the path's first leg (decreasing y)
        sp = spd[:, 0]
        hd32 = float(np.float32(-math.pi / 2))
        for k, v in ((1, 2.0), (2, y), (3, sp * math.cos(hd32)), (4, sp * math.sin(hd32)), (5, hd32), (6, math.sin(hd32)), (7, math.cos(hd32))):
            obs[:, 1, k] = np.where(pick, v, obs[:, 1, k])
    return (torch.from_numpy(obs.astype(np.float32)),
            torch.from_numpy(rs.astype(np.float32)).reshape(B, 1),
            torch.from_numpy(has))
