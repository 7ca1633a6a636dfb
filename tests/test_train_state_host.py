"""CPU: training-state files (train_state.py) -- round trip of everything `train()` restores, the atomic write, the
refusals of a run that cannot continue the saved one (raised before any GPU work), the CLI flags and the recognition of a
plain `state_dict` as weights only."""
import csv
import os

import pytest
import torch

from crowdnav_dsrnn_b200 import Config, train_state
from crowdnav_dsrnn_b200 import train as train_mod
from crowdnav_dsrnn_b200.model import Policy
from crowdnav_dsrnn_b200.spaces import crowd_spaces
from crowdnav_dsrnn_b200.storage import SRNNRolloutStorage

N, H, T = 6, 3, 4


class _Engine:
    """CrowdEngine's get_state / set_state on CPU tensors."""

    def __init__(self, seed):
        g = torch.Generator().manual_seed(seed)
        self.st = {"robot": torch.randn(N, 9, generator=g), "humans": torch.randn(N, H, 9, generator=g),
                   "belief": torch.randn(N, H, 5, generator=g), "extras": torch.randn(N, 4, generator=g),
                   "counters": torch.randint(0, 1000, (N, 4), generator=g, dtype=torch.int32),
                   "episode_return": torch.randn(N, generator=g), "groups": torch.randn(N, 10, 4, generator=g)}

    def get_state(self):
        return {k: v.clone() for k, v in self.st.items()}

    def set_state(self, **fields):
        for k, v in fields.items():
            self.st[k] = torch.as_tensor(v).clone()


def _config(**train):
    cfg = Config(human_num=H)
    cfg.training.num_processes = N
    cfg.ppo.num_steps = T
    for k, v in train.items():
        setattr(cfg.training, k, v)
    return cfg


def _run(seed):
    """Policy + Adam with moments + storage + engine, all on the CPU, filled from `seed`."""
    torch.manual_seed(seed)
    cfg = _config()
    obs, act = crowd_spaces(H)
    policy = Policy(obs.spaces, act, base="srnn", base_kwargs=cfg)
    opt = torch.optim.Adam(policy.parameters(), lr=1e-3, eps=1e-5)
    for p in policy.parameters():
        p.grad = torch.randn_like(p)
    opt.step()
    rollouts = SRNNRolloutStorage(T, N, obs.spaces, act, 128, 256, keep_hidden_history=False)
    for buf in list(rollouts.obs.values()) + list(rollouts.recurrent_hidden_states.values()) + [rollouts.masks, rollouts.bad_masks]:
        buf.copy_(torch.randn_like(buf))
    return cfg, policy, opt, rollouts, _Engine(seed)


def _save(tmp_path, j=3, seed=1, keys=None):
    cfg, policy, opt, rollouts, engine = _run(seed)
    keys = keys if keys is not None else train_state.run_keys(cfg, N, 1, False)
    path = train_state.save(str(tmp_path / "checkpoints"), j, (j + 1) * N * T, keys, policy, opt, engine, rollouts, "cpu")
    return path, (cfg, policy, opt, rollouts, engine)


def _same(a, b):
    if torch.is_tensor(a):
        return torch.is_tensor(b) and a.dtype == b.dtype and torch.equal(a, b)
    if isinstance(a, dict):
        return isinstance(b, dict) and sorted(a, key=str) == sorted(b, key=str) and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return a == b


def test_round_trip_restores_everything(tmp_path):
    path, (_, policy, opt, rollouts, engine) = _save(tmp_path, j=3, seed=1)
    assert os.path.basename(path) == "00003.state.pt"
    assert sorted(os.listdir(tmp_path / "checkpoints")) == ["00003.state.pt", "00003.state.rank0.pt"]
    rng = torch.get_rng_state()
    want_perm = torch.randperm(N)                      # what the next update would draw

    kind, shared, shard = train_state.load(path)
    assert kind == "state" and shared["update"] == 3 and shared["total_steps"] == 4 * N * T and shard["rank"] == 0
    _, policy2, opt2, rollouts2, engine2 = _run(seed=2)   # a fresh process: other weights, moments, envs, generator
    train_state.restore(shared, shard, policy2, opt2, engine2, rollouts2, "cpu")
    assert _same(policy.state_dict(), policy2.state_dict())
    assert _same(opt.state_dict(), opt2.state_dict())
    assert _same(engine.get_state(), engine2.get_state())
    for k in rollouts.obs:
        assert torch.equal(rollouts.obs[k][0], rollouts2.obs[k][0])
    for k in rollouts.recurrent_hidden_states:
        assert torch.equal(rollouts.recurrent_hidden_states[k][0], rollouts2.recurrent_hidden_states[k][0])
    assert torch.equal(rollouts.masks[0], rollouts2.masks[0]) and torch.equal(rollouts.bad_masks[0], rollouts2.bad_masks[0])
    assert torch.equal(torch.get_rng_state(), rng) and torch.equal(torch.randperm(N), want_perm)
    # Adam continues from the restored moments exactly as the original would
    for p, q in zip(policy.parameters(), policy2.parameters()):
        p.grad = torch.full_like(p, 0.5)
        q.grad = torch.full_like(q, 0.5)
    opt.step()
    opt2.step()
    assert _same(policy.state_dict(), policy2.state_dict())


def test_every_tensor_is_stored_on_the_cpu(tmp_path):
    path, _ = _save(tmp_path)
    _, shared, shard = train_state.load(path)
    seen = []

    def walk(x):
        if torch.is_tensor(x):
            seen.append(x.device.type)
        elif isinstance(x, dict):
            [walk(v) for v in x.values()]
        elif isinstance(x, (list, tuple)):
            [walk(v) for v in x]
    walk(shared)
    walk(shard)
    assert seen and set(seen) == {"cpu"}


def test_atomic_write_shows_no_final_name_until_complete(tmp_path, monkeypatch):
    final = str(tmp_path / "00000.state.pt")
    real_save = torch.save
    seen = []

    def checking_save(obj, f):
        seen.append(os.path.exists(final))
        real_save(obj, f)
        seen.append(os.path.exists(final))
    monkeypatch.setattr(torch, "save", checking_save)
    train_state.atomic_save({"x": torch.arange(5)}, final)
    assert seen == [False, False] and os.path.exists(final)
    assert torch.equal(torch.load(final)["x"], torch.arange(5))

    # a write that dies half way leaves neither the final name nor its temporary file behind
    def dying_save(obj, f):
        f.write(b"partial")
        raise KeyboardInterrupt
    monkeypatch.setattr(torch, "save", dying_save)
    other = str(tmp_path / "00001.state.pt")
    with pytest.raises(KeyboardInterrupt):
        train_state.atomic_save({"x": torch.arange(5)}, other)
    assert sorted(os.listdir(tmp_path)) == ["00000.state.pt"]


def _changed(field):
    """(config, world, deterministic) of a run that differs from the saved one in `field` alone."""
    cfg, world, det = _config(resume=True), 1, False
    if field == "envs_per_rank":
        cfg.training.num_processes = N + 2
    elif field == "human_num":
        cfg.sim.human_num = H + 1
    elif field == "num_steps":
        cfg.ppo.num_steps = T + 1
    elif field == "kinematics":
        cfg.action_space.kinematics = "unicycle"
    elif field == "env_config_hash":
        cfg.humans.policy = "social_force"
    elif field == "deterministic":
        cfg.training.cuda_deterministic = det = True
    elif field == "world_size":
        world = 2
    return cfg, world, det


@pytest.mark.parametrize("field", train_state.KEYS)
def test_each_refusal_names_its_field(tmp_path, field):
    path, _ = _save(tmp_path)
    cfg, world, det = _changed(field)
    _, shared, _ = train_state.load(path)
    with pytest.raises(train_state.TrainStateMismatch, match=field) as e:
        train_state.check_keys(shared["keys"], train_state.run_keys(cfg, cfg.training.num_processes, world, det))
    assert e.value.field == field
    if field != "world_size":
        # train() refuses before it builds anything on a device: here on a CPU-only run it would otherwise fail later,
        # in the engine constructor, with a different error
        cfg.training.load_path = path
        with pytest.raises(train_state.TrainStateMismatch, match=field):
            train_mod.train(cfg, "cpu", num_updates=1, output_dir=str(tmp_path / "out"), log=None)
        assert not os.path.exists(tmp_path / "out")


def test_same_run_passes_the_checks(tmp_path):
    path, _ = _save(tmp_path)
    kind, shared, _ = train_state.load(path)
    train_state.check_keys(shared["keys"], train_state.run_keys(_config(), N, 1, False))


def test_a_changed_env_setting_changes_the_hash():
    base = train_state.env_config_hash(_config(), N, 1)
    assert base == train_state.env_config_hash(_config(), N, 1)
    for section, name, value in (("env", "seed", 7), ("reward", "success_reward", 5), ("robot", "FOV", 0.5),
                                 ("sim", "group_human", True)):
        cfg = _config()
        setattr(getattr(cfg, section), name, value)
        assert train_state.env_config_hash(cfg, N, 1) != base, (section, name)


def test_reference_state_dict_is_weights_only(tmp_path):
    cfg, policy, *_ = _run(3)
    path = str(tmp_path / "27776.pt")
    torch.save(policy.state_dict(), path)          # the format of %.5i.pt and of the shipped checkpoints
    kind, sd, shard = train_state.load(path)
    assert kind == "weights" and shard is None and _same(dict(policy.state_dict()), dict(sd))


def test_shards_and_foreign_files_are_refused(tmp_path):
    path, _ = _save(tmp_path)
    with pytest.raises(ValueError, match="shard of rank 0"):
        train_state.load(train_state.rank_path(path, 0))
    with pytest.raises(FileNotFoundError, match="rank 1"):
        train_state.load(path, rank=1)
    other = str(tmp_path / "list.pt")
    torch.save([torch.zeros(2)], other)
    with pytest.raises(ValueError, match="neither"):
        train_state.load(other)


def test_resume_without_load_path_is_refused():
    with pytest.raises(ValueError, match="load_path"):
        train_mod.train(_config(resume=True), "cpu", num_updates=1, output_dir=None, log=None)


def test_cli_flags_map_to_the_config(monkeypatch):
    seen = []
    monkeypatch.setattr(train_mod, "train", lambda cfg, *a, **k: seen.append(cfg))
    train_mod.main(["--envs", "8", "--num_updates", "1", "--save-state", "--resume", "run/checkpoints/00004.state.pt"])
    train_mod.main(["--envs", "8", "--num_updates", "1"])
    a, b = (c.training for c in seen)
    assert a.save_train_state is True and a.resume is True and a.load_path == "run/checkpoints/00004.state.pt"
    assert getattr(b, "save_train_state", False) is False and b.resume is False and b.load_path is None


def test_progress_rows_after_the_resumed_update_are_dropped(tmp_path):
    path = str(tmp_path / "progress.csv")
    with open(path, "w", newline="") as f:
        w = csv.writer(f)
        w.writerow(["misc/nupdates", "misc/total_timesteps", "fps"])
        for j in range(6):
            w.writerow([j, (j + 1) * 10, 1])
    train_mod._drop_progress_after(path, 3)
    with open(path, newline="") as f:
        rows = list(csv.DictReader(f))
    assert [int(r["misc/nupdates"]) for r in rows] == [0, 1, 2, 3]


def _two_rank_worker(rank, world, port, root, ret):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cfg, policy, opt, rollouts, engine = _run(seed=10 + rank)     # each rank owns other envs
    keys = train_state.run_keys(cfg, N, world, False)
    path = train_state.save(os.path.join(root, "checkpoints"), 5, 6 * N * world * T, keys, policy, opt, engine, rollouts,
                            "cpu", rank=rank, world=world)
    ret["files%d" % rank] = sorted(os.listdir(os.path.join(root, "checkpoints")))   # after the barrier: every file is there
    kind, shared, shard = train_state.load(path, rank)
    ret["ok%d" % rank] = kind == "state" and shard["rank"] == rank and not _diff(shard["env"], engine.get_state()) and \
        shared["keys"]["world_size"] == world
    dist.destroy_process_group()


def _diff(a, b):
    return [k for k in a if not torch.equal(a[k], b[k])]


def test_two_ranks_write_their_own_shards(tmp_path):
    """world_size = 2 over gloo: rank 0 writes the shared file, every rank its own shard, and nobody returns before all
    files are in place; each rank reads back its own envs."""
    import socket

    import torch.multiprocessing as mp

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ret = mp.Manager().dict()
    mp.spawn(_two_rank_worker, args=(2, port, str(tmp_path), ret), nprocs=2, join=True)
    files = ["00005.state.pt", "00005.state.rank0.pt", "00005.state.rank1.pt"]
    assert ret["files0"] == files and ret["files1"] == files
    assert ret["ok0"] and ret["ok1"]
