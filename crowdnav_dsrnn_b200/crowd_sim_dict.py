"""`CrowdSimDict`: the single-env gym-style view (crowd_sim/envs/crowd_sim_dict.py:12-271)
over the batched CUDA engine with N = 1.  Same construction protocol as the
reference's make_env thunk (envs.py:47-75): `CrowdSimDict()` -> `.configure(config)`
-> set `.thisSeed`, `.nenv`, `.phase` -> `.reset()` / `.step(action)`.
"""
import numpy as np
import torch

from .engine import CrowdEngine
from .envs import LazyInfos
from .render import check_mode, check_size
from .spaces import crowd_spaces


class CrowdSimDict(object):
    metadata = {}

    def __init__(self, device="cuda"):
        self.device = torch.device(device)
        self.config = None
        self.robot = None
        self.thisSeed = None
        self.nenv = None
        self.phase = None
        self.test_case = None
        self.render_axis = None
        self.render_figure = None
        self._engine = None
        self.observation_space = None
        self.action_space = None

    def configure(self, config):
        self.config = config
        self.time_step = config.env.time_step
        self.time_limit = config.env.time_limit
        self.human_num = config.sim.human_num
        self.observation_space, self.action_space = crowd_spaces(self.human_num)
        from types import SimpleNamespace
        self.robot = SimpleNamespace(time_step=config.env.time_step, v_pref=config.robot.v_pref,
                                     radius=config.robot.radius, kinematics=config.action_space.kinematics)

    def seed(self, seed=None):   # gym.Env.seed is a no-op for this env (envs.py:75)
        return [seed]

    def close(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None

    def _ensure(self):
        if self.config is None or self.robot is None:
            raise AttributeError("robot has to be set!")   # crowd_sim_dict.py:132-133
        if self._engine is None:
            nenv = 1 if self.nenv is None else int(self.nenv)
            seed = self.config.env.seed if self.thisSeed is None else int(self.thisSeed)
            phase = self.phase or ("train" if nenv > 1 else "test")
            self._engine = CrowdEngine(self.config, 1, self.device, phase=phase, seed=seed, nenv=nenv)
        return self._engine

    @property
    def global_time(self):
        steps = int(self._ensure().get_state()["counters"][0, 0].item())
        t = 0
        for _ in range(steps):
            t += self.time_step
        return t

    @staticmethod
    def _host_obs(buf):
        return {"robot_node": buf.robot_node[0].cpu().numpy(), "temporal_edges": buf.temporal_edges[0].cpu().numpy(),
                "spatial_edges": buf.spatial_edges[0].cpu().numpy()}

    def reset(self, phase="train", test_case=None):
        eng = self._ensure()
        if self.test_case is not None:
            test_case = self.test_case
        if test_case is not None:
            st = eng.get_state()
            st["counters"][:, 2] = int(test_case)
            eng.set_state(counters=st["counters"])
        return self._host_obs(eng.reset())

    def render(self, mode="human", size=256):
        """The env's frame as numpy uint8 [size, size, 3] (mode="rgb_array" only; drawn on the GPU)."""
        check_mode(mode)
        check_size(size)
        return self._ensure().render(size=size)[0].cpu().numpy()

    def step(self, action, update=True):
        eng = self._ensure()
        a = torch.as_tensor(np.asarray(action, dtype=np.float32).reshape(1, 2), device=self.device)
        buf = eng.step(a, auto_reset=False)
        infos = LazyInfos(buf, bool(self.config.test.side_preference), 0.0)
        info = infos[0]
        info.pop("episode", None)      # the Monitor wrapper adds it, not the env
        return self._host_obs(buf), float(buf.reward[0].item()), bool(buf.done[0].item()), info
