"""CPU: the host mirror of the env launchers' launch shapes (tests/env_launch_shapes.py) at the B200's 148 SMs, and the
tiling of a sampled state to benchmark-sized batches.  The GPU tests (test_gpu_env_scale.py) rely on both to claim which
kernel path each of their cases runs."""
import numpy as np
import pytest

from crowdnav_dsrnn_b200 import Config, abi
from oracle import state_sampler
import env_launch_shapes as S

SMS = S.B200_SMS


@pytest.mark.parametrize("m,g", [(0, 4), (1, 4), (4, 4), (5, 8), (8, 8), (9, 16), (16, 16), (17, 32), (19, 32), (31, 32)])
def test_pick_group(m, g):
    assert S.pick_group(m) == g


def test_step_shape_production_rule_from_4736_envs_at_h20():
    # H = 20: G = 32, 8 lane groups, ~2 rounds of solves -> E = 8; the small-batch rule applies below 8 * 4 * 148 = 4736
    assert S.step_shape(4735, 20, SMS)["small_batch"] and S.step_shape(4735, 20, SMS)["E"] == 7
    for n in (4736, 16384, 16384 + 5, 65536):
        sh = S.step_shape(n, 20, SMS)
        assert (sh["G"], sh["E"], sh["small_batch"]) == (32, 8, False), n
    assert S.step_shape(2048, 20, SMS)["E"] == 3             # the H = 20 batches of test_gpu_crowd_step.py


def test_step_shape_grid_and_partial_last_cta():
    sh = S.step_shape(16384, 20, SMS)
    assert (sh["grid"], sh["last"]) == (2048, 8)
    sh = S.step_shape(16384 + 5, 20, SMS)
    assert (sh["grid"], sh["last"]) == (2049, 5)
    sh = S.step_shape(1024, 10, SMS)                          # c2: G = 16, E = 8 -> small batch, 1024 // 592 = 1
    assert (sh["G"], sh["E"], sh["grid"], sh["last"]) == (16, 1, 1024, 1)
    sh = S.step_shape(16, 5, SMS)                             # c1
    assert (sh["G"], sh["E"], sh["grid"]) == (4, 1, 16)


def test_step_shape_seq_form():
    # one solve per thread: E = 256 // H, small batches below E * 2 * SMs envs
    sh = S.step_shape(16384, 20, SMS, form="seq")
    assert (sh["E"], sh["small_batch"], sh["grid"]) == (12, False, 1366)
    assert sh["last"] == 16384 - 1365 * 12
    assert S.step_shape(1024, 10, SMS, form="seq")["E"] == 3
    assert S.step_shape(16, 5, SMS, form="seq")["E"] == 1


def test_envs_per_cta_knob_is_clamped_to_the_shared_memory_default():
    assert S.step_envs_per_cta_limit(20) == 43 and S.step_envs_per_cta_limit(32) == 27
    for e in (1, 3, 7, 8, 13, 32, 43):
        sh = S.step_shape(16384 + 5, 20, SMS, envs_per_cta=e)
        assert sh["E"] == e and sh["smem"] <= S.SMEM_DEFAULT
    for e in (44, 46, 64):
        sh = S.step_shape(16384 + 5, 20, SMS, envs_per_cta=e)
        assert sh["E"] == 43 and sh["smem"] <= S.SMEM_DEFAULT
        assert e * 20 * S.STEP_SMEM_PER_HUMAN + S.STEP_SMEM_SCRATCH + S.STEP_SMEM_STATIC > S.SMEM_DEFAULT   # unclamped
    assert S.step_shape(16384, 20, SMS, envs_per_cta=0)["E"] == 8        # out of range: ignored
    assert S.step_shape(16384, 20, SMS, envs_per_cta=65)["E"] == 8
    # the default shape fits at every H
    for h in range(1, 33):
        for rv in (False, True):
            if h + rv <= 32:
                assert S.step_shape(65536, h, SMS, robot_visible=rv)["smem"] <= S.SMEM_DEFAULT, (h, rv)


def test_reset_grids_and_strides():
    assert S.reset_grid(16384, "live") == 16384
    assert S.reset_grid(16384, "spare") == 16384
    assert S.reset_grid(16384, "sync") == 592 and S.reset_grid(512, "sync") == 512
    assert S.reset_grid(16384, "list") == 1184 and S.reset_grid(512, "list") == 512
    assert S.strided_iterations(593, 592) == 2 and S.strided_iterations(592, 592) == 1
    assert S.strided_iterations(1185, 1184) == 2 and S.strided_iterations(0, 1184) == 0


def test_robot_act_partial_last_cta():
    sh = S.robot_act_shape(16384 + 3, 20)
    assert (sh["G"], sh["per_cta"], sh["last"]) == (32, 8, 3)
    sh = S.robot_act_shape(1027, 5)
    assert (sh["G"], sh["per_cta"], sh["last"]) == (8, 32, 3)
    sh = S.robot_act_shape(1024, 5)
    assert sh["last"] == sh["per_cta"]


def test_state_layout_is_256_aligned_and_ordered():
    off, total = S.state_layout(16384 + 5, 20)
    vals = list(off.values())
    assert vals == sorted(vals) and all(v % 256 == 0 for v in vals) and total % 256 == 0
    assert off["hum_gr"] == ((16 * (16384 + 5) * 20 + 255) // 256) * 256
    assert total > off["sp_grp"] + 16 * 8 * (16384 + 5) - 256


def test_tile_state_gives_every_tile_its_own_counters():
    cfg = abi.flatten_config(Config(human_num=3), 64, phase="train")
    inp = state_sampler.sample(cfg, 16, seed=1)
    t = S.tile_state(inp, 16 * 4 + 5)
    for k, v in t.items():
        assert v.shape == (69,) + inp[k].shape[1:] and v.dtype == inp[k].dtype and v.flags.c_contiguous, k
    for k in ("robot", "humans", "belief", "extras", "action"):
        assert np.array_equal(t[k][16:32], inp[k]) and np.array_equal(t[k][64:], inp[k][:5]), k
    c = t["counters"]
    assert np.array_equal(c[:16], inp["counters"])
    assert np.array_equal(c[:, [0, 3]], inp["counters"][np.arange(69) % 16][:, [0, 3]])      # step count, scenario: kept
    for k in range(1, 5):
        blk = c[16 * k:16 * (k + 1)]
        src = inp["counters"][:len(blk)]
        assert np.array_equal(blk[:, 2], src[:, 2] + k * 100003) and np.array_equal(blk[:, 1], src[:, 1] + k)
    # an env and its copies in the other tiles never share a case counter
    assert len(np.unique(c[:, 2])) == len(np.unique(inp["counters"][:, 2])) * 4 + len(np.unique(inp["counters"][:5, 2]))
