"""TEST INFRASTRUCTURE -- host restatement of the model-based robots' action (robot.policy = 'orca' / 'social_force').

For every env the robot's state row is the self and the H belief rows last_human_states (px, py, vx, vy, r) are the
others, in human index order:
  * ORCA: the C oracle's own single solve `oracle_orca_one` (the set-up of crowd_nav/policy/orca.py:64-139 on the
    restated RVO2), called once per env;
  * social force: SOCIAL_FORCE.predict (crowd_nav/policy/social_force.py:11-63) in Python floats, term for term in the
    order of the C oracle's human branch (libm exp / sqrt, no contraction), narrowed to float32 at the end.
"""
import math

import numpy as np

from crowdnav_dsrnn_b200 import abi
from oracle import crowd_oracle

PX, PY, VX, VY, RAD, GX, GY, VPREF = range(8)


def social_force(cfg, self9, others5):
    try:
        return _social_force(cfg, self9, others5)
    except ZeroDivisionError:               # robot on its goal or on an other's position: the reference's action is nan
        return np.array([np.nan, np.nan], np.float32)


def _social_force(cfg, self9, others5):
    s = [float(x) for x in self9]
    gdx, gdy = s[GX] - s[PX], s[GY] - s[PY]
    gdist = math.sqrt(gdx * gdx + gdy * gdy)
    vp = s[VPREF]
    cdx = cfg.sf_KI * ((gdx / gdist) * vp - s[VX])
    cdy = cfg.sf_KI * ((gdy / gdist) * vp - s[VY])
    ivx = ivy = 0.0
    for o in others5:
        ddx, ddy = s[PX] - float(o[0]), s[PY] - float(o[1])
        dist = math.sqrt(ddx * ddx + ddy * ddy)
        f = cfg.sf_A * math.exp((s[RAD] + float(o[4]) - dist) / cfg.sf_B)
        ivx += f * (ddx / dist)
        ivy += f * (ddy / dist)
    nvx = s[VX] + (cdx + ivx) * cfg.time_step
    nvy = s[VY] + (cdy + ivy) * cfg.time_step
    nrm = math.sqrt(nvx * nvx + nvy * nvy)
    if nrm > vp:
        return np.array([nvx / nrm * vp, nvy / nrm * vp], np.float32)
    return np.array([nvx, nvy], np.float32)


def robot_act(cfg, state, policy):
    """Action [N, 2] float32 of a model-based robot ("orca" / "social_force" or abi.POLICY_*) for every env of an
    oracle state (crowd_oracle.OracleState)."""
    code = abi.ROBOT_POLICIES[policy] if isinstance(policy, str) else int(policy)
    out = np.zeros((state.n, 2), np.float32)
    for e in range(state.n):
        if code == abi.POLICY_SOCIAL_FORCE:
            out[e] = social_force(cfg, state.robot[e], state.belief[e])
        else:
            out[e] = crowd_oracle.orca_one(cfg, state.robot[e], state.belief[e])
    return out
