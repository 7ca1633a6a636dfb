"""numpy restatement of the frame of cn_env_render (crowdnav_dsrnn_b200/csrc/render.cu, kernel K7).

Every predicate is the kernel's: the same float32 operations in the same order, without contraction (the kernel is built
with -fmad=false and numpy never fuses).  Next to each frame comes a float64 "margin" per pixel: the smallest distance
(metres) of the pixel centre from the boundary of any shape that is tested there (disc edges, the lines of the FOV wedge
and of the heading sector).  A pixel whose margin is tiny can legitimately differ where the kernel and numpy round a
transcendental (cos / sin of the heading) differently; every other pixel must match exactly.

Palette and marker sizes are read from include/crowdnav_b200.h (the CN_RENDER_* macros), the one place the kernel also
takes them from.
"""
import math
import os
import re

import numpy as np

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "crowdnav_b200.h")
HOLONOMIC = 0
f32 = np.float32


def constants(header=HEADER):
    """CN_RENDER_* macros of the header: {name without the prefix: int or float}."""
    out = {}
    for name, val in re.findall(r"#define\s+CN_RENDER_(\w+)\s+([0-9A-Fa-fx.]+)", open(header).read()):
        out[name] = int(val, 16) if val.lower().startswith("0x") else (float(val) if "." in val else int(val))
    return out


K = constants()


def rgb_bytes(c):
    return np.array([(c >> 16) & 0xFF, (c >> 8) & 0xFF, c & 0xFF], dtype=np.uint8)


def pixel_centres(square_width, size):
    """(x [1, S], y [S, 1]) float32 pixel centres: row 0 at the top, +y up."""
    scale, half = f32(square_width / size), f32(square_width * 0.5)
    j = np.arange(size, dtype=np.float32)
    x = (j + f32(0.5)) * scale - half
    y = half - (j + f32(0.5)) * scale
    return x[None, :], y[:, None]


def heading(kinematics, vx, vy, theta):
    """Unit heading vector in float32: (vx, vy) / |(vx, vy)| for a holonomic robot ((1, 0) at zero speed), (cos th, sin th)
    rounded from float64 otherwise."""
    if kinematics == HOLONOMIC:
        vx, vy = f32(vx), f32(vy)
        n = np.sqrt(vx * vx + vy * vy)
        return (vx / n, vy / n) if n > f32(0.0) else (f32(1.0), f32(0.0))
    return f32(math.cos(float(f32(theta)))), f32(math.sin(float(f32(theta))))


def _disc(x, y, cx, cy, r):
    """(inside, margin) of the disc test dx * dx + dy * dy <= r * r."""
    cx, cy, r = f32(cx), f32(cy), f32(r)
    dx, dy = x - cx, y - cy
    inside = dx * dx + dy * dy <= r * r
    margin = np.abs(np.hypot(x.astype(np.float64) - float(cx), y.astype(np.float64) - float(cy)) - float(r))
    return inside, margin


def _wedge(x, y, ox, oy, fx, fy, c_h, s_h):
    """(inside, margin) of the wedge test c_h * |cross| <= s_h * along around the unit vector f."""
    ox, oy = f32(ox), f32(oy)
    dx, dy = x - ox, y - oy
    a = dx * fx + dy * fy
    c = np.abs(dy * fx - dx * fy)
    inside = c_h * c <= s_h * a
    # |c_h |cross| - s_h along| = |d| |sin(angle - h)|: the distance to the nearer boundary ray, or less
    dx64, dy64 = x.astype(np.float64) - float(ox), y.astype(np.float64) - float(oy)
    a64 = dx64 * float(fx) + dy64 * float(fy)
    c64 = np.abs(dy64 * float(fx) - dx64 * float(fy))
    margin = np.abs(float(c_h) * c64 - float(s_h) * a64)
    return inside, margin


def frame(kinematics, robot_fov, square_width, robot, humans, visible=None, size=256):
    """One frame.  robot [9] and humans [H, 9] in the layout of CrowdEngine.get_state (px, py, vx, vy, radius, gx, gy,
    v_pref, theta); visible: bitmask int (bit i = human i inside the FOV) or None (all inside).
    Returns (rgb uint8 [S, S, 3], margin float64 [S, S])."""
    x, y = pixel_centres(square_width, size)
    shape = (size, size)
    x, y = np.broadcast_to(x, shape), np.broadcast_to(y, shape)
    col = np.full(shape, K["RGB_BACKGROUND"], dtype=np.int64)
    margin = np.full(shape, np.inf)
    robot = np.asarray(robot, dtype=np.float32)
    humans = np.asarray(humans, dtype=np.float32).reshape(-1, 9)
    rx, ry, rr, gx, gy = robot[0], robot[1], robot[4], robot[5], robot[6]
    fx, fy = heading(kinematics, robot[2], robot[3], robot[8])
    if robot_fov < 2.0 * math.pi:
        inside, m = _wedge(x, y, rx, ry, fx, fy, f32(math.cos(robot_fov / 2.0)), f32(math.sin(robot_fov / 2.0)))
        col[inside] = K["RGB_FOV"]
        margin = np.minimum(margin, m)
    inside, m = _disc(x, y, gx, gy, f32(K["GOAL_RADIUS"]))
    col[inside] = K["RGB_GOAL"]
    margin = np.minimum(margin, m)
    for i, h in enumerate(humans):
        inside, m = _disc(x, y, h[0], h[1], h[4])
        seen = visible is None or (int(visible) >> i) & 1
        col[inside] = K["RGB_HUMAN_IN"] if seen else K["RGB_HUMAN_OUT"]
        margin = np.minimum(margin, m)
    inside, m = _disc(x, y, rx, ry, rr)
    margin = np.minimum(margin, m)
    sector, m = _wedge(x, y, rx, ry, fx, fy, f32(math.cos(K["HEADING_HALF"])), f32(math.sin(K["HEADING_HALF"])))
    col[inside] = K["RGB_ROBOT"]
    col[inside & sector] = K["RGB_HEADING"]
    margin = np.minimum(margin, np.where(inside, m, np.inf))       # the sector decides inside the robot disc only
    rgb = np.stack([(col >> 16) & 0xFF, (col >> 8) & 0xFF, col & 0xFF], axis=-1).astype(np.uint8)
    return rgb, margin


def frames(kinematics, robot_fov, square_width, state, env_ids, visible_mask=None, size=256):
    """Frames of `env_ids` from a get_state() dict of numpy arrays; an id outside [0, N) gives the invalid colour (margin
    inf).  visible_mask: [N] bitmasks or None.  Returns (rgb [k, S, S, 3], margin [k, S, S])."""
    n = state["robot"].shape[0]
    rgb = np.empty((len(env_ids), size, size, 3), dtype=np.uint8)
    margin = np.empty((len(env_ids), size, size))
    for k, e in enumerate(env_ids):
        e = int(e)
        if not 0 <= e < n:
            rgb[k] = rgb_bytes(K["RGB_INVALID"])
            margin[k] = np.inf
            continue
        vis = None if visible_mask is None else int(np.asarray(visible_mask).astype(np.int64)[e] & 0xFFFFFFFF)
        rgb[k], margin[k] = frame(kinematics, robot_fov, square_width, state["robot"][e], state["humans"][e], vis, size)
    return rgb, margin
