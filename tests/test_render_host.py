"""CPU: the numpy restatement of the renderer (oracle/render_oracle.py) on hand-built scenes, so that it and the kernel
cannot be wrong together; baselines' tile_images layout; the PNG writer; argument errors raised before any library call."""
import math
import re
import struct
import zlib

import numpy as np
import pytest

from crowdnav_dsrnn_b200 import abi
from crowdnav_dsrnn_b200.crowd_sim_dict import CrowdSimDict
from crowdnav_dsrnn_b200.envs import CrowdVecEnv
from crowdnav_dsrnn_b200.render import check_mode, check_size, tile_images, write_png
from oracle import render_oracle as ro

K = ro.K
L = 10.0                       # sim.square_width of the default config
FAR = 1000.0                   # somewhere outside every frame


def rgb(name):
    return ro.rgb_bytes(K["RGB_" + name])


def mask_of(img, name):
    return np.all(img == rgb(name), axis=-1)


def robot(px=FAR, py=FAR, vx=0.0, vy=0.0, r=0.3, gx=FAR, gy=FAR, theta=0.0):
    return np.array([px, py, vx, vy, r, gx, gy, 1.0, theta], dtype=np.float32)


def human(px, py, r):
    return np.array([px, py, 0, 0, r, 0, 0, 1, 0], dtype=np.float32)


def centres(size):
    """Exact float64 pixel centres (pitch and offsets are dyadic for L = 10 and S = 2^k, so no rounding happens)."""
    j = np.arange(size, dtype=np.float64)
    return (j + 0.5) * (L / size) - L / 2, L / 2 - (j + 0.5) * (L / size)


def test_header_is_the_one_place_of_palette_and_sizes():
    text = open(ro.HEADER).read()
    assert re.search(r"CN_RENDER_RGB_BACKGROUND", text)
    for name, value in abi.RENDER_RGB.items():
        assert K["RGB_" + name.upper()] == value, name
    assert K["GOAL_RADIUS"] == abi.RENDER_GOAL_RADIUS and K["HEADING_HALF"] == abi.RENDER_HEADING_HALF
    assert (K["MIN_SIZE"], K["MAX_SIZE"], K["SIZE_MULTIPLE"]) == (abi.RENDER_MIN_SIZE, abi.RENDER_MAX_SIZE,
                                                                  abi.RENDER_SIZE_MULTIPLE)
    assert len(set(abi.RENDER_RGB.values())) == len(abi.RENDER_RGB)        # every layer is distinguishable


@pytest.mark.parametrize("cx,cy,r", [(0.0, 0.0, 0.5), (1.25, -2.5, 0.3), (-4.9, 4.9, 0.4), (0.15625, 0.15625, 0.7)])
def test_single_human_covers_the_expected_pixels(cx, cy, r):
    S = 32
    img, _ = ro.frame(abi.HOLONOMIC, 2 * math.pi, L, robot(), [human(cx, cy, r)], None, S)
    xs, ys = centres(S)
    want = (xs[None, :] - cx) ** 2 + (ys[:, None] - cy) ** 2 <= np.float64(np.float32(r)) ** 2
    assert np.array_equal(mask_of(img, "HUMAN_IN"), want)
    assert np.array_equal(mask_of(img, "BACKGROUND"), ~want)


def test_a_disc_through_one_pixel_centre_colours_that_pixel_only():
    S = 64
    xs, ys = centres(S)
    img, _ = ro.frame(abi.HOLONOMIC, 2 * math.pi, L, robot(), [human(xs[7], ys[3], 0.01)], 0, S)
    hit = np.argwhere(mask_of(img, "HUMAN_OUT"))
    assert hit.tolist() == [[3, 7]]


@pytest.mark.parametrize("r", [0.2, 0.3, 0.55, 1.3])
def test_disc_area_is_pi_r_squared_within_one_pixel_perimeter(r):
    S = 256
    pitch = L / S
    img, _ = ro.frame(abi.HOLONOMIC, 2 * math.pi, L, robot(), [human(0.37, -0.81, r)], None, S)
    area = mask_of(img, "HUMAN_IN").sum() * pitch * pitch
    assert abs(area - math.pi * r * r) <= 2 * math.pi * r * pitch


def _fov_at(img, S, x, y):
    xs, ys = centres(S)
    return bool(mask_of(img, "FOV")[np.argmin(np.abs(ys - y)), np.argmin(np.abs(xs - x))])


def test_fov_wedge_follows_the_velocity_of_a_holonomic_robot():
    S = 128
    fov = math.pi * 0.5                     # robot.FOV = 0.5: +-45 degrees
    img, _ = ro.frame(abi.HOLONOMIC, fov, L, robot(0.0, 0.0, vx=0.0, vy=0.8, gx=FAR), [human(FAR, FAR, 0.3)], None, S)
    assert _fov_at(img, S, 0.0, 3.0) and _fov_at(img, S, 1.5, 3.0) and _fov_at(img, S, -1.5, 3.0)
    assert not _fov_at(img, S, 3.0, 1.0) and not _fov_at(img, S, -3.0, 1.0) and not _fov_at(img, S, 0.0, -3.0)
    # at zero speed the heading is (1, 0), as detect_visible's atan2(0, 0) = 0
    img, _ = ro.frame(abi.HOLONOMIC, fov, L, robot(0.0, 0.0), [human(FAR, FAR, 0.3)], None, S)
    assert _fov_at(img, S, 3.0, 0.0) and not _fov_at(img, S, -3.0, 0.0) and not _fov_at(img, S, 0.0, 3.0)
    share = mask_of(img, "FOV").mean()
    assert abs(share - 0.25) < 0.02                # a right-angle wedge from the centre covers a quarter of the square


def test_fov_wedge_follows_theta_of_a_unicycle_robot_and_is_absent_at_fov_2():
    S = 128
    img, _ = ro.frame(abi.UNICYCLE, math.pi * 0.5, L, robot(1.0, 1.0, vx=1.0, vy=0.0, theta=math.pi), [human(FAR, FAR, 0.3)],
                      None, S)
    assert _fov_at(img, S, -2.0, 1.0) and not _fov_at(img, S, 4.0, 1.0)        # theta wins over the velocity
    img, _ = ro.frame(abi.UNICYCLE, math.pi * 2.0, L, robot(1.0, 1.0, theta=math.pi), [human(FAR, FAR, 0.3)], None, S)
    assert not mask_of(img, "FOV").any()


def test_heading_sector_points_along_the_heading():
    S = 256
    img, _ = ro.frame(abi.UNICYCLE, 2 * math.pi, L, robot(0.0, 0.0, r=1.0, theta=math.pi / 2), [], None, S)
    xs, ys = centres(S)
    heading = mask_of(img, "HEADING")
    rows, cols = np.nonzero(heading)
    assert heading.any() and ys[rows].min() >= -1e-9 and np.abs(xs[cols]).max() < 1.0 * math.sin(0.5) + L / S
    assert mask_of(img, "ROBOT").sum() > 4 * heading.sum()


def test_draw_order_later_layers_cover_earlier_ones():
    S = 64
    xs, ys = centres(S)
    # goal under human 0 under human 1 under the robot, all overlapping at the centre pixel of row 31, column 31
    c = (xs[31], ys[31])
    r0 = robot(c[0] + 0.2, c[1], r=0.1, gx=c[0] - 0.1, gy=c[1])
    hs = [human(c[0], c[1], 0.5), human(c[0] + 0.1, c[1], 0.4)]
    for bits, top in ((0b10, "HUMAN_IN"), (0b01, "HUMAN_OUT")):
        img, _ = ro.frame(abi.HOLONOMIC, 2 * math.pi, L, r0, hs, bits, S)
        assert np.array_equal(img[31, 31], rgb(top))                    # human 1 over human 0 and the goal
        assert mask_of(img, "ROBOT").any() or mask_of(img, "HEADING").any()
        assert not mask_of(img, "GOAL").any()                           # the goal lies under human 0
    img, _ = ro.frame(abi.HOLONOMIC, 2 * math.pi, L, r0, hs[:0], None, S)
    assert mask_of(img, "GOAL").any()


def test_invalid_ids_and_margins():
    S = 32
    st = {"robot": robot(0.0, 0.0)[None], "humans": np.stack([human(1.0, 1.0, 0.3)])[None]}
    img, margin = ro.frames(abi.HOLONOMIC, math.pi, L, st, [0, -1, 1], np.array([1]), S)
    assert np.all(img[1] == rgb("INVALID")) and np.all(img[2] == rgb("INVALID")) and np.isinf(margin[1]).all()
    assert margin[0].min() >= 0 and np.isfinite(margin[0]).any()


def test_tile_images_layout():
    frames = np.arange(1, 6, dtype=np.uint8)[:, None, None, None] * np.ones((5, 2, 3, 3), dtype=np.uint8)
    img = tile_images(frames)
    assert img.shape == (3 * 2, 2 * 3, 3)                   # rows = ceil(sqrt(5)) = 3, cols = ceil(5 / 3) = 2
    cells = [[int(img[r * 2, c * 3, 0]) for c in range(2)] for r in range(3)]
    assert cells == [[1, 2], [3, 4], [5, 0]]                # row-major, the unused cell zero
    assert tile_images(frames[:1]).shape == (2, 3, 3)
    assert tile_images(np.zeros((64, 4, 4, 3), np.uint8)).shape == (32, 32, 3)


def test_png_writer_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, size=(5, 7, 3), dtype=np.uint8)
    p = tmp_path / "x.png"
    write_png(str(p), img)
    data = p.read_bytes()
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    w, h = struct.unpack(">II", data[16:24])
    assert (w, h) == (7, 5)
    n = struct.unpack(">I", data[33:37])[0]
    assert data[37:41] == b"IDAT"
    raw = np.frombuffer(zlib.decompress(data[41:41 + n]), dtype=np.uint8).reshape(5, 1 + 7 * 3)
    assert (raw[:, 0] == 0).all() and np.array_equal(raw[:, 1:].reshape(5, 7, 3), img)


@pytest.mark.parametrize("size", [0, 16, 30, 40, 100, 2064, 4096, 256.0, "256", True, None])
def test_bad_sizes_are_refused(size):
    with pytest.raises((ValueError, TypeError)):
        check_size(size)


def test_good_sizes_pass():
    assert [check_size(s) for s in (32, 48, 256, 1024, 2048, np.int64(64))] == [32, 48, 256, 1024, 2048, 64]


def test_argument_errors_come_before_any_library_call():
    """No GPU, no engine: the modes and sizes are refused by Python first (the objects below have no engine at all)."""
    vec = object.__new__(CrowdVecEnv)
    for mode in ("human", "rgb", None):
        with pytest.raises(NotImplementedError):
            vec.render(mode=mode)
    with pytest.raises(ValueError):
        vec.render(mode="rgb_array", size=100)
    sim = CrowdSimDict(device="cpu")
    with pytest.raises(NotImplementedError):
        sim.render()
    with pytest.raises(ValueError):
        sim.render(mode="rgb_array", size=33)
    with pytest.raises(NotImplementedError):
        check_mode("human")
