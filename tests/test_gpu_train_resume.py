"""GPU: resumable training (train_state.py).  A deterministic run that stops after an update and is continued by a fresh
`train()` from its training-state file writes the same checkpoints, the same progress rows and ends in the same training
state (envs, rollout storage, optimizer, both generators) as a run that was never interrupted; `load_path` naming a
plain state_dict starts from exactly those weights; in the default (atomic) mode a resumed run continues within the
native update's usual tolerance."""
import csv
import math
import os

import numpy as np
import pytest
import torch

from crowdnav_dsrnn_b200 import Config
from crowdnav_dsrnn_b200.train import train

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = {
    "holonomic_h5": dict(human_num=5),
    "holonomic_h20_fov": dict(human_num=20, **{"robot.FOV": 0.5}),
    "unicycle_h5": dict(human_num=5, kinematics="unicycle"),                     # theta, desiredVelocity
    "group_h10": dict(human_num=10, **{"sim.group_human": True}),                # the episode's circle groups
    "mixed_policies_h8": dict(human_num=8, **{"humans.random_policy_changing": True}),   # per-human ORCA / social force
}


def _config(case, deterministic=True, **training):
    spec = dict(CASES[case])
    cfg = Config(human_num=spec.pop("human_num"), kinematics=spec.pop("kinematics", "holonomic"))
    for key, value in spec.items():
        section, name = key.split(".")
        setattr(getattr(cfg, section), name, value)
    cfg.training.num_processes = 256
    cfg.ppo.num_steps = 30
    cfg.training.cuda_deterministic = deterministic
    cfg.training.save_interval = 1
    cfg.training.log_interval = 1
    cfg.training.save_train_state = True
    for name, value in training.items():
        setattr(cfg.training, name, value)
    return cfg


def _resumed(case, load_path, deterministic=True):
    return _config(case, deterministic, resume=True, load_path=str(load_path))


def _ckpt(run, name):
    return torch.load(os.path.join(run, "checkpoints", name), map_location="cpu", weights_only=True)


def _progress(run):
    with open(os.path.join(run, "progress.csv"), newline="") as f:
        return [{k: v for k, v in r.items() if k != "fps"} for r in csv.DictReader(f)]


def _same(a, b, where=""):
    """Bit equality of nested state (tensors, dicts, lists, scalars); returns the paths that differ."""
    if torch.is_tensor(a):
        return [] if torch.is_tensor(b) and a.dtype == b.dtype and torch.equal(a, b) else [where]
    if isinstance(a, dict):
        if not isinstance(b, dict) or sorted(a, key=str) != sorted(b, key=str):
            return [where + "{keys}"]
        return [d for k in a for d in _same(a[k], b[k], "%s/%s" % (where, k))]
    if isinstance(a, (list, tuple)):
        if len(a) != len(b):
            return [where + "[len]"]
        return [d for i, (x, y) in enumerate(zip(a, b)) for d in _same(x, y, "%s[%d]" % (where, i))]
    return [] if a == b or (isinstance(a, float) and math.isnan(a) and math.isnan(b)) else [where]


def _strip(rows):
    return [{k: v for k, v in r.items() if k != "fps"} for r in rows]


@pytest.mark.parametrize("case", sorted(CASES))
def test_resumed_deterministic_run_equals_uninterrupted_run(tmp_path, case):
    run_a, run_b = str(tmp_path / "a"), str(tmp_path / "b")
    kw = dict(log=None, native_update=True)
    _, hist_a = train(_config(case), DEV, num_updates=4, output_dir=run_a, **kw)
    _, hist_b1 = train(_config(case), DEV, num_updates=2, output_dir=run_b, **kw)
    assert sum(r["episodes"] for r in hist_b1) > 0, "no episode ended before the resume point: resets are not exercised"
    policy, hist_b2 = train(_resumed(case, os.path.join(run_b, "checkpoints", "00001.state.pt")), DEV, num_updates=4,
                            output_dir=run_b, **kw)
    assert [r["misc/nupdates"] for r in hist_b2] == [2, 3]
    for name in ("00002.pt", "00003.pt"):
        sd_a, sd_b = _ckpt(run_a, name), _ckpt(run_b, name)
        assert sorted(sd_a) == sorted(sd_b) and not _same(sd_a, sd_b), name
    assert not _same(_strip(hist_a[2:]), _strip(hist_b2))       # losses, success, collision, timeout, episodes, reward
    assert _progress(run_a) == _progress(run_b)                  # every column but fps, rows 0..3 in order
    # the training state after the last update: envs (all CnStateView fields), rollout slot 0, optimizer, generators
    for name in ("00003.state.pt", "00003.state.rank0.pt"):
        diff = _same(_ckpt(run_a, name), _ckpt(run_b, name))
        assert not diff, (name, diff[:10])


def test_weights_only_resume_starts_from_those_weights(tmp_path):
    """load_path naming a shipped-format state_dict: a fresh run from exactly those weights (lr = 0 keeps them through one
    update, so checkpoint 00000 must hold them bit for bit)."""
    w = np.load(os.path.join(ROOT, "tests", "golden", "weights_holonomic_27776.npz"))
    shipped = {k: torch.from_numpy(w[k].copy()) for k in w.files}
    path = str(tmp_path / "27776.pt")
    torch.save(shipped, path)
    cfg = _config("holonomic_h5", lr=0.0, resume=True, load_path=path)
    cfg.training.save_train_state = False
    _, hist = train(cfg, DEV, num_updates=1, output_dir=str(tmp_path / "run"), log=None, native_update=True)
    assert [r["misc/nupdates"] for r in hist] == [0]
    sd = _ckpt(str(tmp_path / "run"), "00000.pt")
    assert sorted(sd) == sorted(shipped) and not _same(shipped, sd)
    assert sorted(os.listdir(tmp_path / "run" / "checkpoints")) == ["00000.pt"]


def test_resume_in_default_mode_continues_within_tolerance(tmp_path):
    """Without training.cuda_deterministic the update adds split-K partial sums with atomics: a resumed update starts from
    the saved state bit for bit and differs from the uninterrupted one only by that summation order."""
    run_a, run_c = str(tmp_path / "a"), str(tmp_path / "c")
    kw = dict(log=None, native_update=True)
    _, hist_a = train(_config("holonomic_h5", deterministic=False), DEV, num_updates=3, output_dir=run_a, **kw)
    _, hist_c = train(_resumed("holonomic_h5", os.path.join(run_a, "checkpoints", "00001.state.pt"), deterministic=False),
                      DEV, num_updates=3, output_dir=run_c, **kw)
    assert len(hist_c) == 1 and hist_c[0]["misc/nupdates"] == 2
    a, c = hist_a[2], hist_c[0]
    assert all(math.isfinite(c[k]) for k in ("loss/value_loss", "loss/policy_loss", "loss/policy_entropy"))
    assert c["episodes"] == a["episodes"]        # the rollout of update 2 runs on the restored weights and envs
    assert abs(c["loss/value_loss"] - a["loss/value_loss"]) <= 1e-3 * abs(a["loss/value_loss"])
    assert abs(c["loss/policy_loss"] - a["loss/policy_loss"]) <= 1e-4
    assert abs(c["loss/policy_entropy"] - a["loss/policy_entropy"]) <= 1e-5
    # checkpoint numbering continues in the new directory
    assert sorted(os.listdir(os.path.join(run_c, "checkpoints"))) == ["00002.pt", "00002.state.pt", "00002.state.rank0.pt"]
