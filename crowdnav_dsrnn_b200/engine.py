"""Batched crowd-simulation engine: N envs resident in HBM, stepped by the CUDA
kernels behind the C ABI (include/crowdnav_b200.h).  torch is used only for
device memory and streams.

This is the object `make_vec_envs` (envs.py) and `CrowdSimDict`
(crowd_sim_dict.py) wrap; it replaces the reference's
ShmemVecEnv -> _subproc_worker -> CrowdSimDict.step/reset chain
(pytorchBaselines/a2c_ppo_acktr/shmem_vec_env.py:97-107,160-168;
crowd_sim/envs/crowd_sim_dict.py:105-271).
"""
import ctypes as C

import torch

from . import _lib, abi
from .render import check_size as _check_render_size


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class StepBuffers:
    """One set of per-step outputs (torch-owned device tensors in the reference's shapes)."""

    # per-step records a caller may keep beyond the next step (infos): carved out of ONE block so that a single
    # device-side clone snapshots them all (envs.LazyInfos).  reward | done come last and next to each other: they are what
    # the reference-facing step() brings to the host, in one copy (envs.CrowdVecEnv.step_wait)
    INFO_FIELDS = (("info", torch.float32, abi.INFO_DIM), ("episode_return", torch.float32, 1),
                   ("event", torch.int32, 1), ("scenario", torch.int32, 1), ("episode_length", torch.int32, 1),
                   ("reward", torch.float32, 1), ("done", torch.uint8, 1))
    _ITEMSIZE = {torch.float32: 4, torch.int32: 4, torch.uint8: 1}
    _layouts = {}

    @classmethod
    def info_layout(cls, n):
        """((name, dtype, width, byte offset, byte length), ...), total bytes -- every field starts on a 256-byte boundary."""
        lay = cls._layouts.get(n)
        if lay is None:
            fields, off = [], 0
            for name, dtype, width in cls.INFO_FIELDS:
                nbytes = n * width * cls._ITEMSIZE[dtype]
                fields.append((name, dtype, width, off, nbytes))
                off += (nbytes + 255) & ~255
            lay = cls._layouts[n] = (tuple(fields), off)
        return lay

    @classmethod
    def carve_info(cls, block, n):
        """Typed views (name -> tensor) into an info block."""
        views = {}
        for name, dtype, width, off, nbytes in cls.info_layout(n)[0]:
            v = block[off:off + nbytes].view(dtype)
            views[name] = v.view(n, width) if width > 1 else v
        return views

    @classmethod
    def info_block_bytes(cls, n):
        return cls.info_layout(n)[1]

    @classmethod
    def host_range(cls, n):
        """Byte range of the info block that holds reward | done, and done's offset inside it."""
        lay = {f[0]: f for f in cls.info_layout(n)[0]}
        lo, hi = lay["reward"][3], lay["done"][3] + lay["done"][4]
        return lo, hi, lay["done"][3] - lo

    def __init__(self, n, h, device):
        f32 = dict(dtype=torch.float32, device=device)
        self.n = n
        self.robot_node = torch.zeros(n, 1, 7, **f32)
        self.temporal_edges = torch.zeros(n, 1, 2, **f32)
        self.spatial_edges = torch.zeros(n, h, 2, **f32)
        self.visible_mask = torch.zeros(n, dtype=torch.int32, device=device)
        self.info_block = torch.zeros(self.info_block_bytes(n), dtype=torch.uint8, device=device)
        for name, view in self.carve_info(self.info_block, n).items():
            setattr(self, name, view)
        lo, hi, _ = self.host_range(n)
        self.host_bytes = self.info_block[lo:hi]           # reward | done as one contiguous byte range
        self.goal_changed = torch.zeros(n, dtype=torch.int32, device=device)
        self.not_done = torch.ones(n, 1, **f32)            # 1 - done: the masks of the next Policy.act
        self.obs_struct = abi.CnObsOut(_ptr(self.robot_node), _ptr(self.temporal_edges), _ptr(self.spatial_edges),
                                       _ptr(self.visible_mask))
        self.step_struct = abi.CnStepOut(self.obs_struct, _ptr(self.reward), _ptr(self.done), _ptr(self.event),
                                         _ptr(self.scenario), _ptr(self.info), _ptr(self.episode_return),
                                         _ptr(self.episode_length), _ptr(self.goal_changed), _ptr(self.not_done))

    def obs(self):
        return {"robot_node": self.robot_node, "temporal_edges": self.temporal_edges,
                "spatial_edges": self.spatial_edges}


class CrowdEngine:
    STATE_FIELDS = ("robot", "humans", "belief", "extras", "counters", "episode_return", "groups")

    def __init__(self, config, n_envs, device, phase=None, seed=None, env_id_offset=0, nenv=None, **tries):
        device = torch.device(device)
        if device.type != "cuda":
            raise _lib.CrowdNavLibraryError("CrowdEngine needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.lib = _lib.load()
        self.device = device
        self.n, self.h = int(n_envs), int(config.sim.human_num)
        self.config = config
        self.cfg = abi.flatten_config(config, n_envs, phase=phase, seed=seed, env_id_offset=env_id_offset,
                                      nenv=nenv, **tries)
        nbytes = self.lib.cn_env_state_bytes(C.byref(self.cfg), self.n)
        if nbytes == 0:
            _lib.check(-1, "cn_env_state_bytes")
        self.state = torch.zeros(nbytes, dtype=torch.uint8, device=device)
        handle = C.c_void_p()
        index = device.index if device.index is not None else torch.cuda.current_device()
        self.device_index = index
        _lib.check(self.lib.cn_env_create(C.byref(self.cfg), self.n, index, _ptr(self.state), nbytes, C.byref(handle)),
                   "cn_env_create")
        self.handle = handle
        # double-buffered so the observation returned by step k stays valid while step k+1 runs
        self.bufs = [StepBuffers(self.n, self.h, device), StepBuffers(self.n, self.h, device)]
        self.cur = 0
        self.launches = 0

    def close(self):
        if getattr(self, "handle", None):
            for ref in self.__dict__.pop("_refill_policies", []):      # forwards must not call into a destroyed env
                policy = ref()
                if policy is not None and policy.__dict__.get("_refill_engine") is self:
                    policy.start_refill_of(None)
            self.lib.cn_env_destroy(self.handle)
            self.handle = None

    __del__ = close

    def _stream(self):
        return _lib.raw_stream(self.device_index)

    # ------------------------------------------------------------------ API
    def reset(self, mask=None):
        """CrowdSimDict.reset on every env (or where mask != 0). Returns the StepBuffers holding the obs."""
        self.cur ^= 1
        b = self.bufs[self.cur]
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            prev = self.bufs[self.cur ^ 1]
            for name in ("robot_node", "temporal_edges", "spatial_edges", "visible_mask"):
                getattr(b, name).copy_(getattr(prev, name))
        _lib.check(self.lib.cn_env_reset(self.handle, _ptr(mask), C.byref(b.obs_struct), self._stream()), "cn_env_reset")
        self.launches += self.lib.cn_env_last_launches(self.handle)
        return b

    def step(self, action, auto_reset=True, defer_refill=False):
        """CrowdSimDict.step on every env; action [N,2] float32 on the device.  `defer_refill`: the spare-episode refill is
        started by the next forward (Policy.start_refill_of) instead of right behind the step kernel."""
        if action.device != self.device or action.dtype != torch.float32 or not action.is_contiguous():
            action = action.to(device=self.device, dtype=torch.float32).contiguous()
        if action.numel() != 2 * self.n:
            raise ValueError("action must have shape [%d, 2]" % self.n)
        self.cur ^= 1
        b = self.bufs[self.cur]
        mode = (2 if defer_refill else 1) if auto_reset else 0
        _lib.check(self.lib.cn_env_step(self.handle, _ptr(action), C.byref(b.step_struct), mode, self._stream()), "cn_env_step")
        self.launches += self.lib.cn_env_last_launches(self.handle)
        return b

    def robot_act(self, policy, out=None):
        """Action of a model-based robot on every env from the running state: ORCA.predict / SOCIAL_FORCE.predict with the
        robot as self and the belief rows last_human_states as the others (cn_env_robot_act) -> device float32 [N, 2],
        the velocities to pass to step().  `policy`: "orca" / "social_force" (or abi.POLICY_*), on a holonomic engine
        whatever config.robot.policy is.  `out` (contiguous float32 [N, 2] on this device) gives the result a static
        address (CUDA graphs)."""
        code = abi.ROBOT_POLICIES.get(policy, policy) if isinstance(policy, str) else int(policy)
        if code not in abi.ROBOT_POLICIES.values():
            raise ValueError("policy must be one of %s, got %r" % (sorted(abi.ROBOT_POLICIES), policy))
        dev = torch.device("cuda", self.device_index)
        if out is None:
            out = torch.empty(self.n, 2, dtype=torch.float32, device=dev)
        elif out.dtype != torch.float32 or out.device != dev or tuple(out.shape) != (self.n, 2) or not out.is_contiguous():
            raise ValueError("out must be a contiguous float32 tensor [%d, 2] on %s" % (self.n, dev))
        _lib.check(self.lib.cn_env_robot_act(self.handle, code, _ptr(out), self._stream()), "cn_env_robot_act")
        self.launches += self.lib.cn_env_last_launches(self.handle)
        return out

    def join(self):
        """Make the current stream wait for the spare-episode refill forked by the last reset()/step() (the library joins it
        by itself at the next call; an explicit join is needed at the end of a CUDA-graph capture)."""
        _lib.check(self.lib.cn_env_join(self.handle, self._stream()), "cn_env_join")

    def observe(self):
        self.cur ^= 1
        b = self.bufs[self.cur]
        _lib.check(self.lib.cn_env_observe(self.handle, C.byref(b.obs_struct), self._stream()), "cn_env_observe")
        self.launches += self.lib.cn_env_last_launches(self.handle)
        return b

    def render(self, env_ids=None, size=256, out=None):
        """rgb_array frames of envs `env_ids` (None: all; a list, or an int32 device tensor for a capturable call) drawn by
        cn_env_render from the running state and the current buffer's visible_mask -> device uint8 [k, size, size, 3].
        `out` (contiguous uint8 [k, size, size, 3] on this device) gives the frames a static address (CUDA graphs; a captured
        render reads the visible_mask of the step buffer that was current at capture).  An id outside [0, N) gives a frame
        of the "invalid" colour."""
        size = _check_render_size(size)
        dev = torch.device("cuda", self.device_index)
        if env_ids is None:
            ids, k = None, self.n
        else:
            ids = env_ids
            if not (torch.is_tensor(ids) and ids.device == dev and ids.dtype == torch.int32 and ids.is_contiguous()):
                ids = torch.as_tensor(env_ids, dtype=torch.int32).to(dev).contiguous()   # allocates: not capturable
            ids = ids.reshape(-1)
            k = ids.numel()
        if out is None:
            out = torch.empty(k, size, size, 3, dtype=torch.uint8, device=dev)
        elif (out.dtype != torch.uint8 or out.device != dev or tuple(out.shape) != (k, size, size, 3)
              or not out.is_contiguous()):
            raise ValueError("out must be a contiguous uint8 tensor [%d, %d, %d, 3] on %s" % (k, size, size, dev))
        _lib.check(self.lib.cn_env_render(self.handle, _ptr(ids), k, _ptr(self.bufs[self.cur].visible_mask), size,
                                          _ptr(out), self._stream()), "cn_env_render")
        self.launches += self.lib.cn_env_last_launches(self.handle)
        return out

    # ------------------------------------------------------------------ state injection / extraction
    def _state_tensors(self):
        f32 = dict(dtype=torch.float32, device=self.device)
        return {
            "robot": torch.zeros(self.n, 9, **f32), "humans": torch.zeros(self.n, self.h, 9, **f32),
            "belief": torch.zeros(self.n, self.h, 5, **f32), "extras": torch.zeros(self.n, 4, **f32),
            "counters": torch.zeros(self.n, 4, dtype=torch.int32, device=self.device),
            "episode_return": torch.zeros(self.n, **f32),
            "groups": torch.zeros(self.n, abi.MAX_GROUPS, 4, **f32),      # group environment: radius, cx, cy, valid
        }

    def get_state(self):
        t = self._state_tensors()
        view = abi.CnStateView(*[_ptr(t[f]) for f in self.STATE_FIELDS])
        _lib.check(self.lib.cn_env_get_state(self.handle, C.byref(view), self._stream()), "cn_env_get_state")
        return t

    def set_state(self, **fields):
        keep = {}
        for f in self.STATE_FIELDS:
            v = fields.get(f)
            if v is not None:
                dt = torch.int32 if f == "counters" else torch.float32
                v = torch.as_tensor(v).to(device=self.device, dtype=dt).contiguous()
            keep[f] = v
        view = abi.CnStateView(*[_ptr(keep[f]) for f in self.STATE_FIELDS])
        _lib.check(self.lib.cn_env_set_state(self.handle, C.byref(view), self._stream()), "cn_env_set_state")
        torch.cuda.current_stream(self.device).synchronize()  # `keep` must outlive the copy kernel
