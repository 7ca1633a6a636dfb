"""GPU: cn_env_render (K7, csrc/render.cu) against the numpy restatement oracle/render_oracle.py, and the public
render(mode="rgb_array") / get_images API around it.

Every pixel must equal the restatement, except pixels whose margin (float64 distance of the pixel centre from a shape
boundary) is below MARGIN metres; those may differ only where the kernel's fp64 cos / sin of the heading rounds to
another float than the host's, and fewer than MAX_SHARE of a frame may differ.  Axis-aligned scenes match exactly."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from crowdnav_dsrnn_b200 import Config, _lib, abi
from crowdnav_dsrnn_b200.crowd_sim_dict import CrowdSimDict
from crowdnav_dsrnn_b200.engine import CrowdEngine
from crowdnav_dsrnn_b200.envs import CrowdVecEnv
from oracle import render_oracle as ro

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
MARGIN = 1e-4          # metres
MAX_SHARE = 1e-3
CN_ERR_ARG = -1


def make_cfg(kin="holonomic", H=5, fov=2.0, group=False, social_force=False):
    cfg = Config(kinematics=kin, human_num=H)
    cfg.robot.FOV = fov
    cfg.robot.visible = True
    if group:
        cfg.sim.group_human = True
    if social_force:
        cfg.humans.policy = "social_force"
    return cfg


def warm_engine(cfg, n, steps=7, seed=3):
    """An engine some steps into its episodes, with the visible mask of the current observation."""
    eng = CrowdEngine(cfg, n, DEV, phase="train", seed=seed)
    eng.reset()
    g = torch.Generator(device="cpu").manual_seed(seed)
    for _ in range(steps):
        eng.step((torch.rand(n, 2, generator=g) * 2 - 1).to(DEV), auto_reset=True)
    return eng


def oracle_frames(eng, ids, size, mask=True):
    st = {k: v.cpu().numpy() for k, v in eng.get_state().items()}
    vm = eng.bufs[eng.cur].visible_mask.cpu().numpy() if mask else None
    return ro.frames(eng.cfg.kinematics, eng.cfg.robot_fov, eng.cfg.square_width, st, ids, vm, size)


def assert_frames(got, want, margin, exact=False):
    got = got.cpu().numpy() if torch.is_tensor(got) else got
    assert got.shape == want.shape
    diff = np.any(got != want, axis=-1)
    if exact:
        assert not diff.any(), "%d pixels differ in an axis-aligned scene" % int(diff.sum())
        return
    bad = diff & (margin >= MARGIN)
    assert not bad.any(), "%d pixels differ at margin >= %g m (first at %s)" % (int(bad.sum()), MARGIN, np.argwhere(bad)[0])
    per_frame = diff.reshape(diff.shape[0], -1).mean(axis=1)
    assert per_frame.max() < MAX_SHARE, "%.2e of a frame differs" % per_frame.max()


@pytest.mark.parametrize("kin", ["holonomic", "unicycle"])
@pytest.mark.parametrize("fov", [0.5, 2.0])
@pytest.mark.parametrize("H", [1, 5, 20, 31])
def test_kernel_matches_the_restatement(kin, fov, H):
    n = 24
    eng = warm_engine(make_cfg(kin, H, fov), n)
    for size, ids in ((32, list(range(n))), (256, [5, 0, 23, 5, 11, 17, 2]), (1024, [9])):
        got = eng.render(ids, size=size)
        want, margin = oracle_frames(eng, ids, size)
        assert_frames(got, want, margin)
    eng.close()


@pytest.mark.parametrize("opts", [dict(group=True, H=8), dict(social_force=True, H=5), dict(group=True, social_force=True, H=16)])
def test_group_and_social_force_crowds(opts):
    n = 32
    eng = warm_engine(make_cfg("unicycle", fov=0.7, **opts), n, steps=12)
    ids = list(range(n))
    got = eng.render(ids, size=256)
    want, margin = oracle_frames(eng, ids, 256)
    assert_frames(got, want, margin)
    eng.close()


def test_overlapping_humans_and_the_frame_edge():
    """Injected state: humans overlapping each other, the robot and all four frame edges; huge, tiny and zero radii."""
    H, n = 20, 6
    eng = CrowdEngine(make_cfg("holonomic", H, 0.8), n, DEV, phase="train", seed=1)
    eng.reset()
    st = eng.get_state()
    half = eng.cfg.square_width / 2
    g = torch.Generator(device="cpu").manual_seed(7)
    hum = st["humans"].cpu()
    hum[:, :, 0] = (torch.rand(n, H, generator=g) * 2 - 1) * 1.5
    hum[:, :, 1] = (torch.rand(n, H, generator=g) * 2 - 1) * 1.5
    hum[:, :, 4] = 0.2 + torch.rand(n, H, generator=g) * 0.8
    hum[:, 0, 0:2] = torch.tensor([half, 0.0])                  # on the edges and corners
    hum[:, 1, 0:2] = torch.tensor([-half - 0.2, half - 0.1])
    hum[:, 2, 0:2] = torch.tensor([0.3, -half])
    hum[:, 3, 0:2] = torch.tensor([half + 0.05, half + 0.05])
    hum[:, 4, 4] = 3 * half                                     # covers the whole frame
    hum[:, 5, 4] = 0.0
    hum[:, 6, 4] = 1e-3
    hum[1, 4, 4] = 0.3
    rob = st["robot"].cpu()
    rob[:, 0:2] = torch.tensor([0.2, -0.1])
    rob[:, 2:4] = torch.tensor([0.6, -0.3])
    rob[2, 0:2] = torch.tensor([half - 0.1, -half + 0.1])
    eng.set_state(humans=hum, robot=rob)
    eng.observe()
    ids = list(range(n))
    for size in (32, 256, 1024):
        got = eng.render(ids, size=size)
        want, margin = oracle_frames(eng, ids, size)
        assert_frames(got, want, margin)
    eng.close()


@pytest.mark.parametrize("kin", ["holonomic", "unicycle"])
def test_axis_aligned_scene_matches_exactly(kin):
    """Heading (1, 0) and dyadic positions and radii: nothing is rounded differently, so every pixel matches."""
    H, n = 5, 3
    eng = CrowdEngine(make_cfg(kin, H, 0.5), n, DEV, phase="train", seed=1)
    eng.reset()
    st = eng.get_state()
    rob = torch.zeros(n, 9)
    rob[:, 0:4] = torch.tensor([0.5, -1.25, 1.0, 0.0])
    rob[:, 4] = 0.375
    rob[:, 5:7] = torch.tensor([4.0, 2.5])
    rob[:, 7] = 1.0
    hum = st["humans"].cpu()
    for i in range(H):
        hum[:, i, 0:2] = torch.tensor([-3.0 + 1.25 * i, 0.75 * i - 1.0])
        hum[:, i, 4] = 0.25 + 0.125 * i
    eng.set_state(robot=rob, humans=hum)
    eng.observe()
    for size in (32, 256):
        got = eng.render([2, 0, 1], size=size)
        want, margin = oracle_frames(eng, [2, 0, 1], size)
        assert_frames(got, want, margin, exact=True)
    eng.close()


def test_env_ids_subset_unsorted_duplicates_and_out_of_range():
    n = 10
    eng = warm_engine(make_cfg("unicycle", 5, 0.5), n)
    ids = [7, 2, 2, -1, 9, n, 0, 2 ** 31 - 1, -2 ** 31, 3]
    got = eng.render(ids, size=64)
    want, margin = oracle_frames(eng, ids, 64)
    assert_frames(got, want, margin)
    invalid = torch.tensor(ro.rgb_bytes(abi.RENDER_RGB["invalid"]), device=DEV)
    for k in (3, 5, 7, 8):
        assert bool((got[k] == invalid).all())
    assert torch.equal(got[1], got[2])
    # a device tensor of ids, and the default (all envs, in order)
    dev_ids = torch.tensor(ids, dtype=torch.int32, device=DEV)
    assert torch.equal(eng.render(dev_ids, size=64), got)
    everything = eng.render(size=64)
    assert everything.shape == (n, 64, 64, 3)
    assert torch.equal(everything[7], got[0])
    eng.close()


def test_rendering_does_not_disturb_the_simulation():
    """An engine that renders after every step of a 100-step auto-reset rollout and a twin that never renders produce the
    same outputs and state, bit for bit."""
    cfg = make_cfg("holonomic", 5, 0.6)
    n = 64
    engines = [CrowdEngine(cfg, n, DEV, phase="train", seed=9) for _ in range(2)]
    for e in engines:
        e.reset()
    g = torch.Generator(device="cpu").manual_seed(4)
    fields = ("robot_node", "temporal_edges", "spatial_edges", "visible_mask", "reward", "done", "event", "info",
              "episode_return", "episode_length", "not_done")
    done_seen = 0
    for _ in range(100):
        action = (torch.rand(n, 2, generator=g) * 2 - 1).to(DEV)
        outs = []
        for i, e in enumerate(engines):
            b = e.step(action, auto_reset=True)
            if i == 0:
                e.render(list(range(0, n, 3)), size=128)
            outs.append({f: getattr(b, f).clone() for f in fields})
        for f in fields:
            assert torch.equal(outs[0][f], outs[1][f]), f
        done_seen += int(outs[0]["done"].sum())
    assert done_seen > 0                                       # auto-resets happened
    s0, s1 = (e.get_state() for e in engines)
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k
    for e in engines:
        e.close()


def test_frame_after_an_auto_reset_shows_the_new_episode():
    cfg = make_cfg("holonomic", 5, 2.0)
    n = 64
    eng = CrowdEngine(cfg, n, DEV, phase="train", seed=2)
    eng.reset()
    g = torch.Generator(device="cpu").manual_seed(2)
    S = 256
    pitch = eng.cfg.square_width / S
    for _ in range(200):
        b = eng.step((torch.rand(n, 2, generator=g) * 2 - 1).to(DEV), auto_reset=True)
        done = torch.nonzero(b.done).flatten().tolist()
        if done:
            break
    assert done, "no episode ended in 200 steps"
    frames = eng.render(done, size=S).cpu().numpy()
    node = b.robot_node[done, 0].cpu().numpy()               # the reset observation: the new episode's robot
    robot_colours = (ro.rgb_bytes(abi.RENDER_RGB["robot"]), ro.rgb_bytes(abi.RENDER_RGB["heading"]))
    for k in range(len(done)):
        px, py = node[k, 0], node[k, 1]
        j = int(math.floor((px + eng.cfg.square_width / 2) / pitch))
        i = int(math.floor((eng.cfg.square_width / 2 - py) / pitch))
        assert 0 <= i < S and 0 <= j < S
        assert any(np.array_equal(frames[k, i, j], c) for c in robot_colours), (k, i, j, frames[k, i, j])
    want, margin = oracle_frames(eng, done, S)
    assert_frames(frames, want, margin)
    eng.close()


def test_render_captured_in_a_cuda_graph_equals_the_eager_render():
    cfg = make_cfg("unicycle", 20, 0.5)
    n = 128
    eng = warm_engine(cfg, n)
    ids = torch.tensor([3, 100, 3, 0, 127, 200, 64], dtype=torch.int32, device=DEV)
    out = torch.zeros(len(ids), 256, 256, 3, dtype=torch.uint8, device=DEV)
    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        eng.render(ids, size=256, out=out)                     # warm-up outside the capture
    torch.cuda.current_stream(DEV).wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        eng.render(ids, size=256, out=out)
    out.zero_()
    g = torch.Generator(device="cpu").manual_seed(1)
    for _ in range(3):
        # the graph reads the state as it is at replay time, and the visible mask of the step buffer that was current at
        # capture: two steps bring that buffer back to current
        for _ in range(2):
            eng.step((torch.rand(n, 2, generator=g) * 2 - 1).to(DEV), auto_reset=True)
        graph.replay()
        assert torch.equal(out, eng.render(ids, size=256))
    eng.close()


def test_public_api_shapes():
    cfg = make_cfg("holonomic", 5, 2.0)
    venv = CrowdVecEnv(cfg, 70, DEV, seed=1)
    venv.reset()
    tile = venv.render("rgb_array", size=32)
    assert isinstance(tile, np.ndarray) and tile.dtype == np.uint8 and tile.shape == (8 * 32, 8 * 32, 3)   # 64 envs
    imgs = venv.get_images(size=64)
    assert imgs.is_cuda and imgs.dtype == torch.uint8 and imgs.shape == (70, 64, 64, 3)
    assert np.array_equal(tile[32:64, 64:96], venv.get_images([10], size=32)[0].cpu().numpy())   # row 1, column 2 = env 10
    view = venv.envs[3].env.render(mode="rgb_array")
    assert isinstance(view, np.ndarray) and view.shape == (256, 256, 3)
    assert np.array_equal(view, venv.get_images([3])[0].cpu().numpy())
    with pytest.raises(NotImplementedError):
        venv.render("human")
    with pytest.raises(NotImplementedError):
        venv.envs[0].env.render()
    venv.close()
    small = CrowdVecEnv(cfg, 5, DEV, seed=1)
    small.reset()
    assert small.render("rgb_array", size=48).shape == (3 * 48, 2 * 48, 3)       # rows 3, cols 2, one empty cell
    assert (small.render("rgb_array", size=48)[2 * 48:, 48:] == 0).all()
    small.close()
    sim = CrowdSimDict()
    sim.configure(cfg)
    sim.reset()
    frame = sim.render(mode="rgb_array", size=128)
    assert frame.shape == (128, 128, 3) and frame.dtype == np.uint8
    with pytest.raises(NotImplementedError):
        sim.render(mode="human")
    sim.close()


def test_bad_arguments_are_library_errors_not_crashes():
    eng = warm_engine(make_cfg(), 8, steps=1)
    lib = _lib.load()
    out = torch.zeros(8, 256, 256, 3, dtype=torch.uint8, device=DEV)
    ptr = C.c_void_p(out.data_ptr())
    stream = _lib.raw_stream(0)
    for k, size, rgb in ((8, 30, ptr), (8, 4096, ptr), (8, 0, ptr), (8, 250, ptr), (-1, 256, ptr), (8, 256, None),
                         (9, 256, ptr), (8, 256, C.c_void_p(out.data_ptr() + 3))):
        rc = lib.cn_env_render(eng.handle, None, k, None, size, rgb, stream)
        assert rc == CN_ERR_ARG, (k, size, rc)
        with pytest.raises(_lib.CrowdNavLibraryError):
            _lib.check(rc, "cn_env_render")
    assert lib.cn_env_render(eng.handle, None, 0, None, 256, None, stream) == 0       # k == 0: nothing to do
    assert lib.cn_env_last_launches(eng.handle) == 0
    assert lib.cn_env_render(eng.handle, None, 8, None, 256, ptr, stream) == 0
    assert lib.cn_env_last_launches(eng.handle) == 1
    assert eng.render([], size=64).shape == (0, 64, 64, 3)
    with pytest.raises(ValueError):
        eng.render(size=100)
    with pytest.raises(ValueError):
        eng.render([0, 1], size=64, out=torch.zeros(3, 64, 64, 3, dtype=torch.uint8, device=DEV))
    torch.cuda.synchronize()
    eng.close()
