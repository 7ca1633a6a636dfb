"""`make_vec_envs`: same signature and returned-object contract as
pytorchBaselines/a2c_ppo_acktr/envs.py:106-156 (+ VecPyTorch :208-246 and the
auto-reset worker of shmem_vec_env.py:160-168), but the N envs are ONE batched
simulation resident in HBM and stepped by the CUDA kernels -- no worker
processes, pipes, pickling or host round trips.

Returned object (`CrowdVecEnv`):
  .observation_space.spaces / .action_space / .num_envs
  .reset()            -> dict[str, float32 Tensor on device]
  .step(action[N,2])  -> (obs dict, reward CPU float32 Tensor [N,1], done numpy bool [N], infos)
                         (robot.policy 'orca' / 'social_force': the robot acts by itself and `action` is ignored)
  .step_async / .step_wait / .render(mode="rgb_array") / .get_images / .close
  .venv.envs[0].env   -> object with .global_time .time_step .time_limit .robot.{time_step,v_pref} (evaluation.py:71)
`infos` is a lazy sequence: `infos[i]` builds the reference-shaped dict
({"info": {..., "event": Collision()}, "episode": {"r","l","t"}}) only when it
is indexed or iterated; `.tensors` gives the same data as device tensors for
callers that do not want the host copy.
"""
import time
from types import SimpleNamespace

import numpy as np
import torch

from . import abi
from .engine import CrowdEngine, StepBuffers
from .info import make_event
from .render import check_mode, check_size, tile_images
from .spaces import crowd_spaces


class LazyInfos(object):
    """Sequence of per-env info dicts materialised on access (SURVEY 7, hard part 7)."""

    def __init__(self, buf, side_preference, t0):
        # The engine double-buffers its outputs, so `buf` is overwritten by the step after next.  The reference returns
        # materialised dicts that stay valid for ever (train.py keeps them for logging), so the per-step records are
        # snapshotted here -- one device-side clone of the block they are carved from, no synchronisation.
        # The typed views are carved out of the snapshot on first use: a training loop that never looks at `infos` pays
        # for one clone per step and nothing else.
        self._block, self._n = buf.info_block.clone(), buf.n
        self._tensors = None
        self._side = side_preference
        self._host = None
        self._t0 = t0

    @property
    def tensors(self):
        if self._tensors is None:
            snap = StepBuffers.carve_info(self._block, self._n)
            self._tensors = {k: snap[k] for k in ("event", "scenario", "info", "done", "episode_return", "episode_length")}
        return self._tensors

    def _fetch(self):
        if self._host is None:
            self._host = {k: v.cpu().numpy() for k, v in self.tensors.items()}
        return self._host

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        h = self._fetch()
        row = h["info"][i]
        col = abi.INFO_COLUMNS
        scenario = abi.SCENARIOS[int(h["scenario"][i])]
        step_info = {
            "aggregate_nav_time": int(row[col["aggregate_nav_time"]]),
            "path_violation": int(row[col["path_violation"]]),
            "personal_violation": int(row[col["personal_violation"]]),
            "jerk_cost": float(row[col["jerk_cost"]]),
            "dist_to_goal": float(row[col["dist_to_goal"]]),
            "speed_violation": int(row[col["speed_violation"]]),
            "scenario": scenario,
            "event": make_event(int(h["event"][i]), float(row[col["dmin"]])),
        }
        if self._side:
            step_info[scenario] = {"left": int(row[col["side_left"]]), "right": int(row[col["side_right"]])}
            step_info["separation"] = float(row[col["separation"]])
        info = {"info": step_info}
        if h["done"][i]:  # baselines.bench.Monitor
            info["episode"] = {"r": round(float(h["episode_return"][i]), 6), "l": int(h["episode_length"][i]),
                               "t": round(time.time() - self._t0, 6)}
        return info

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class _EnvView(object):
    """What evaluation.py:71 reaches for through `.venv.envs[0].env`."""

    def __init__(self, vec, index):
        self._vec, self._i = vec, index
        cfg = vec.config
        self.time_step = cfg.env.time_step
        self.time_limit = cfg.env.time_limit
        self.robot = SimpleNamespace(time_step=cfg.env.time_step, v_pref=cfg.robot.v_pref, radius=cfg.robot.radius,
                                     kinematics=cfg.action_space.kinematics)
        self.config = cfg

    @property
    def global_time(self):
        steps = int(self._vec.engine.get_state()["counters"][self._i, 0].item())
        t = 0
        for _ in range(steps):
            t += self.time_step
        return t

    def render(self, mode="human", size=256):
        """This env's frame: numpy uint8 [size, size, 3] (mode="rgb_array" only)."""
        check_mode(mode)
        return self._vec.get_images([self._i], size=size)[0].cpu().numpy()


class CrowdVecEnv(object):
    def __init__(self, config, num_envs, device, seed=0, phase=None, test_case=-1, env_id_offset=0, nenv=None):
        # robot.policy 'orca' / 'social_force': every step first asks the model-based robot for its action
        # (CrowdEngine.robot_act) and the caller's actions are ignored; refused before any CUDA work
        self.robot_policy = abi.robot_policy_of(config)
        self.config = config
        self.num_envs = int(num_envs)
        self.device = torch.device(device)
        self.engine = CrowdEngine(config, self.num_envs, self.device, phase=phase, seed=seed,
                                  env_id_offset=env_id_offset, nenv=nenv)
        self._robot_action = None
        self.observation_space, self.action_space = crowd_spaces(config.sim.human_num)
        self._side = bool(config.test.side_preference)
        self._t0 = time.time()
        self._pending = None
        self._pin_reward = self._pin_done = self._pin_host = None
        self._test_case = test_case
        envs = [SimpleNamespace(env=_EnvView(self, i)) for i in range(min(self.num_envs, 64))]
        self.venv = SimpleNamespace(envs=envs, num_envs=self.num_envs)
        self.envs = envs

    def reset(self):
        if self._test_case is not None and self._test_case >= 0:  # envs.py:61-63: a fixed test case selects the seed
            st = self.engine.get_state()
            st["counters"][:, 2] = int(self._test_case)
            self.engine.set_state(counters=st["counters"])
        return self.engine.reset().obs()

    def step_async(self, actions):
        self._pending = actions

    def _step_engine(self, actions):
        if self.robot_policy is not None:
            if self._robot_action is None:
                self._robot_action = torch.empty(self.num_envs, 2, dtype=torch.float32, device=self.device)
            actions = self.engine.robot_act(self.robot_policy, out=self._robot_action)
        return self.engine.step(actions, auto_reset=True)

    def step_wait(self):
        buf = self._step_engine(self._pending)
        self._pending = None
        # VecPyTorch.step_wait keeps reward on the CPU and done as a numpy array (envs.py:231-239): both cross PCIe in
        # ONE synchronisation through pinned staging buffers (fresh host tensors are returned, like the reference)
        if self._pin_reward is None:
            lo, hi, done_off = StepBuffers.host_range(self.num_envs)
            pin = torch.empty(hi - lo, dtype=torch.uint8)
            if self.device.type == "cuda":
                pin = pin.pin_memory()
            self._pin_host = pin
            self._pin_reward = pin[:4 * self.num_envs].view(torch.float32)
            self._pin_done = pin[done_off:done_off + self.num_envs].numpy()
        self._pin_host.copy_(buf.host_bytes, non_blocking=True)
        infos = LazyInfos(buf, self._side, self._t0)      # its device-side snapshot is enqueued BEFORE the host waits
        if self.device.type == "cuda":
            torch.cuda.current_stream(self.device).synchronize()
        reward = self._pin_reward.clone().unsqueeze(1)
        done = self._pin_done.astype(bool)
        return buf.obs(), reward, done, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def step_device(self, actions):
        """Tensor-native fast path: everything stays on the GPU, nothing is synchronised."""
        buf = self._step_engine(actions)
        return buf.obs(), buf.reward, buf.done, buf

    def get_images(self, env_ids=None, size=256):
        """baselines' VecEnv.get_images, kept on the device: uint8 [k, size, size, 3] of envs `env_ids` (default all),
        drawn by the GPU from the running state (CrowdEngine.render)."""
        return self.engine.render(env_ids, size=size)

    def render(self, mode="human", size=256):
        """baselines' VecEnv.render(mode="rgb_array"): the frames of the envs in `self.envs` (the first min(N, 64)) as one
        numpy [rows * size, cols * size, 3] tile (tile_images layout).  Only "rgb_array" is supported."""
        check_mode(mode)
        check_size(size)
        return tile_images(self.get_images(list(range(len(self.envs))), size=size).cpu().numpy())

    def close(self):
        self.engine.close()


def make_vec_envs(env_name, seed, num_processes, gamma, log_dir, device, allow_early_resets,
                  num_frame_stack=None, config=None, ax=None, test_case=-1, fig=None):
    """Drop-in for envs.py:106-156.  `gamma`, `log_dir`, `allow_early_resets`, `num_frame_stack`, `ax`, `fig`
    are accepted for signature compatibility (they only matter for Box observations / rendering)."""
    if env_name != "CrowdSimDict-v0":
        raise NotImplementedError("only CrowdSimDict-v0 is on the hot path (got %r)" % (env_name,))
    if config is None:
        raise ValueError("config is required")
    return CrowdVecEnv(config, num_processes, device, seed=seed, test_case=test_case)
