"""Training-state files: everything `train()` needs to continue a run after update j in a fresh process.

A `%.5i.pt` checkpoint holds the policy weights only (train.py:326-339 of the reference), which is not enough to continue a
run: Adam's moments, the update index, the envs, the rollout's last observation and hidden state and both random
generators are lost.  With `training.save_train_state` set, `train()` also writes, at every checkpoint and after the
last update, the state as it stands right after `rollouts.after_update()`:

* `<output_dir>/checkpoints/%.5i.state.pt`, shared by all ranks (rank 0 writes it): the policy `state_dict`, the
  optimizer `state_dict`, the update index j, the env-steps so far and the keys a resumed run must match (`KEYS`);
* `<output_dir>/checkpoints/%.5i.state.rank<r>.pt`, one per rank: `CrowdEngine.get_state()` (every field, groups
  included), slot 0 of the rollout storage (observation, both hidden states, masks, bad_masks), the CPU generator state
  (the update's minibatch `randperm`) and the CUDA generator state of the rank's device (action sampling in
  `Policy.act`; None when the run is not on a GPU).

Every tensor is stored on the CPU.  A file is written under a temporary name and renamed when complete, so a job killed
while writing never leaves a file that looks complete.  `training.resume` with `training.load_path` naming a shared file
continues the run with update j + 1; naming a plain `state_dict` (the format of `%.5i.pt` and of the reference's shipped
checkpoints) it loads the weights and starts a fresh run.
"""
import hashlib
import os

import torch

from . import abi

FORMAT = "crowdnav_dsrnn_b200.train_state"
VERSION = 1
# what a resumed run must share with the run that wrote the state, in the order the refusals are checked
KEYS = ("world_size", "envs_per_rank", "human_num", "num_steps", "kinematics", "env_config_hash", "deterministic")


class TrainStateMismatch(ValueError):
    """The state file was written by a run this one cannot continue; `field` names the first key that differs."""

    def __init__(self, field, saved, current):
        super().__init__("cannot resume: %s differs (saved state: %r, this run: %r)" % (field, saved, current))
        self.field, self.saved, self.current = field, saved, current


def shared_path(ckpt_dir, j):
    return os.path.join(ckpt_dir, "%.5i.state.pt" % j)


def rank_path(shared, rank):
    """`<dir>/00007.state.pt` -> `<dir>/00007.state.rank<rank>.pt`."""
    base, ext = os.path.splitext(shared)
    return "%s.rank%d%s" % (base, rank, ext)


def env_config_hash(config, n_envs, world):
    """SHA-256 of the flattened env config the engine of rank 0 is built from: any change to the simulated envs
    (scenarios, rewards, human behaviours, seed, ...) changes it."""
    cfg = abi.flatten_config(config, n_envs, phase="train", seed=config.env.seed, env_id_offset=0, nenv=n_envs * world)
    return hashlib.sha256(bytes(cfg)).hexdigest()


def run_keys(config, n_envs, world, deterministic):
    return {"world_size": int(world), "envs_per_rank": int(n_envs), "human_num": int(config.sim.human_num),
            "num_steps": int(config.ppo.num_steps), "kinematics": str(config.action_space.kinematics),
            "env_config_hash": env_config_hash(config, n_envs, world), "deterministic": bool(deterministic)}


def check_keys(saved, current):
    """Raise TrainStateMismatch naming the first key in KEYS on which the two runs differ."""
    for k in KEYS:
        if saved.get(k) != current[k]:
            raise TrainStateMismatch(k, saved.get(k), current[k])


def _cpu(x):
    if torch.is_tensor(x):
        return x.detach().to("cpu", copy=True)
    if isinstance(x, dict):
        return {k: _cpu(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return type(x)(_cpu(v) for v in x)
    return x


def atomic_save(obj, path):
    """torch.save to `path` through a temporary name in the same directory: `path` appears only once the file is complete."""
    tmp = "%s.tmp%d" % (path, os.getpid())
    try:
        with open(tmp, "wb") as f:
            torch.save(obj, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    except BaseException:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise


def _is_cuda(device):
    return torch.device(device).type == "cuda"


def capture_shared(j, total_steps, keys, actor_critic, optimizer):
    return {"format": FORMAT, "version": VERSION, "kind": "shared", "update": int(j), "total_steps": int(total_steps),
            "keys": dict(keys), "policy": _cpu(actor_critic.state_dict()), "optimizer": _cpu(optimizer.state_dict())}


def capture_rank(j, rank, keys, engine, rollouts, device):
    storage = {"obs": {k: v[0] for k, v in rollouts.obs.items()},
               "hidden": {k: v[0] for k, v in rollouts.recurrent_hidden_states.items()},
               "masks": rollouts.masks[0], "bad_masks": rollouts.bad_masks[0]}
    return {"format": FORMAT, "version": VERSION, "kind": "rank", "update": int(j), "rank": int(rank), "keys": dict(keys),
            "env": _cpu(engine.get_state()), "storage": _cpu(storage),
            "rng_cpu": torch.get_rng_state(), "rng_cuda": torch.cuda.get_rng_state(device) if _is_cuda(device) else None}


def save(ckpt_dir, j, total_steps, keys, actor_critic, optimizer, engine, rollouts, device, rank=0, world=1):
    """Write rank `rank`'s shard and (rank 0) the shared file of update j.  With several ranks every rank must call this;
    nobody returns before every file is in place.  Returns the shared file's path."""
    os.makedirs(ckpt_dir, exist_ok=True)
    path = shared_path(ckpt_dir, j)
    atomic_save(capture_rank(j, rank, keys, engine, rollouts, device), rank_path(path, rank))
    if rank == 0:
        atomic_save(capture_shared(j, total_steps, keys, actor_critic, optimizer), path)
    if world > 1:
        torch.distributed.barrier()
    return path


def is_train_state(obj):
    return isinstance(obj, dict) and obj.get("format") == FORMAT


def load(path, rank=0):
    """Read `training.load_path`.  Returns ("state", shared, shard) for a training-state file (the shard of `rank` is read
    from next to it) or ("weights", state_dict, None) for a plain state_dict.  Anything else is refused."""
    obj = torch.load(path, map_location="cpu", weights_only=True)
    if is_train_state(obj):
        if obj.get("version") != VERSION:
            raise ValueError("%s: training-state format version %r, this build reads %d" % (path, obj.get("version"), VERSION))
        if obj.get("kind") != "shared":
            raise ValueError("%s is the shard of rank %r; pass the shared file (%%.5i.state.pt) as training.load_path"
                             % (path, obj.get("rank")))
        shard_file = rank_path(path, rank)
        if not os.path.exists(shard_file):
            raise FileNotFoundError("%s: the shard of rank %d (%s) is missing" % (path, rank, shard_file))
        shard = torch.load(shard_file, map_location="cpu", weights_only=True)
        if not is_train_state(shard) or shard.get("kind") != "rank" or shard.get("rank") != rank or \
                shard.get("update") != obj["update"] or shard.get("keys") != obj["keys"]:
            raise ValueError("%s does not belong to %s (update %r of rank %d expected)" % (shard_file, path, obj["update"], rank))
        return "state", obj, shard
    if isinstance(obj, dict) and obj and all(isinstance(k, str) and torch.is_tensor(v) for k, v in obj.items()):
        return "weights", obj, None
    raise ValueError("%s is neither a training-state file nor a policy state_dict" % (path,))


def restore(shared, shard, actor_critic, optimizer, engine, rollouts, device):
    """Put a run back where `shared` / `shard` captured it.  Call after every constructor (policy, PPO, envs, storage)
    and after `envs.reset()`: the random generators are restored last, so nothing built afterwards draws from them."""
    actor_critic.load_state_dict(shared["policy"])
    if hasattr(actor_critic, "invalidate_weights"):
        actor_critic.invalidate_weights()
    optimizer.load_state_dict(shared["optimizer"])
    engine.set_state(**shard["env"])
    st = shard["storage"]
    for k, v in st["obs"].items():
        rollouts.obs[k][0].copy_(v)
    for k, v in st["hidden"].items():
        rollouts.recurrent_hidden_states[k][0].copy_(v)
    rollouts.masks[0].copy_(st["masks"])
    rollouts.bad_masks[0].copy_(st["bad_masks"])
    torch.set_rng_state(shard["rng_cpu"])
    if _is_cuda(device):
        torch.cuda.synchronize(device)
        torch.cuda.set_rng_state(shard["rng_cuda"], device)
