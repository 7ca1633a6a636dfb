"""Training driver (SURVEY.md 8(f) rows N1/N3): the loop of the reference's train.py:205-400 on the batched backend.

Per update: `ppo.num_steps` rollout steps (`Policy.act` -> CUDA forward, `CrowdVecEnv.step_device` -> CUDA crowd step, both
device resident, no host synchronisation inside the rollout), `get_value` bootstrap, `compute_returns`, `PPO.update`,
`after_update`; checkpoints are `state_dict`s named `%.5i.pt` under `<output_dir>/checkpoints` (train.py:326-339) and
`progress.csv` has the reference's columns (train.py:363-372).  Episode statistics are reduced on the device
(the reference walks a Python list of info dicts per step, train.py:263-276).

`training.cuda_deterministic` (the reference's switch: its train.py puts cuDNN into deterministic mode) makes a run
reproducible: cuDNN is set to deterministic mode and the native update sums its split-K reductions in a fixed order
(`PPO(deterministic=True)`), so two runs with the same seed write checkpoints with identical tensors.

`training.save_train_state` (`--save-state`) also writes training-state files next to the checkpoints (train_state.py),
and `training.resume` with `training.load_path` (`--resume PATH`) continues a run from one: in deterministic mode the
continued run writes the same checkpoints as a run that was never interrupted.  `load_path` may also name a plain
`state_dict` (a `%.5i.pt` checkpoint or a shipped one): its weights start a fresh run.

Under `torch.distributed` every rank runs this function with its own shard of `training.num_processes` envs
(env ids offset by rank so the episode seeds do not collide) and `PPO` averages the gradients; rank 0 writes artefacts.
"""
import csv
import inspect
import logging
import os
import shutil
import sys
import time

import torch
import torch.distributed as dist

from . import abi
from . import train_state
from .envs import CrowdVecEnv
from .model import Policy
from .ppo import PPO, update_linear_schedule
from .storage import SRNNRolloutStorage


def _rank_world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def write_run_artefacts(config, out_dir):
    """What the reference's train.py writes before the loop starts (train.py:47-75): the config snapshot
    `<out>/configs/train_config.py` (+ `configs/config.py` pointing at the live file, a symlink there) -- test.py re-imports
    it as `<model_dir>.configs.train_config` (test.py:60-98) -- and `<out>/output.log`.  Returns the file logger."""
    cfg_dir = os.path.join(out_dir, "configs")
    os.makedirs(cfg_dir, exist_ok=True)
    try:
        src = inspect.getsourcefile(type(config))
    except TypeError:
        src = None
    if src and os.path.exists(src):
        shutil.copyfile(src, os.path.join(cfg_dir, "train_config.py"))
        link = os.path.join(cfg_dir, "config.py")
        if not os.path.lexists(link):
            os.symlink(os.path.abspath(src), link)
    # the values actually used (the class file above only holds the defaults when the caller edited the instance)
    with open(os.path.join(cfg_dir, "train_config_values.txt"), "w") as f:
        for sec, bag in sorted(vars(config).items()):
            for k, v in sorted(vars(bag).items()) if hasattr(bag, "__dict__") else ():
                f.write("%s.%s = %r\n" % (sec, k, v))
    logger = logging.getLogger("crowdnav_dsrnn_b200.train.%d" % os.getpid())
    logger.setLevel(logging.INFO)
    logger.propagate = False
    for h in list(logger.handlers):
        logger.removeHandler(h)
    handler = logging.FileHandler(os.path.join(out_dir, "output.log"), mode="a" if getattr(config.training, "resume", False) else "w")
    handler.setFormatter(logging.Formatter("%(asctime)s, %(levelname)s: %(message)s", datefmt="%Y-%m-%d %H:%M:%S"))
    logger.addHandler(handler)
    return logger


def _tensorboard_writer(out_dir):
    """TensorBoard scalars of train.py:211,376-386 when the `tensorboard` package is importable (it is optional here)."""
    try:
        from torch.utils.tensorboard import SummaryWriter
    except Exception:  # noqa: BLE001
        return None
    return SummaryWriter(log_dir=os.path.join(out_dir, "events"))


def _resume_source(config, n_envs, world, rank, deterministic):
    """What `training.load_path` holds when `training.resume` is set: None (no resume), ("weights", state_dict, None) or
    ("state", shared, shard) of a training-state file that this run can continue (else TrainStateMismatch)."""
    if not getattr(config.training, "resume", False):
        return None
    path = getattr(config.training, "load_path", None)
    if not path:
        raise ValueError("training.resume is set but training.load_path names no file to resume from")
    source = train_state.load(path, rank)
    if source[0] == "state":
        train_state.check_keys(source[1]["keys"], train_state.run_keys(config, n_envs, world, deterministic))
    return source


def _drop_progress_after(path, last):
    """A resumed run appends to progress.csv: rows the interrupted run wrote after the update it resumes from go first."""
    if not os.path.exists(path):
        return
    with open(path, newline="") as f:
        rows = list(csv.reader(f))
    keep = rows[:1] + [r for r in rows[1:] if r and int(r[0]) <= last]
    if len(keep) != len(rows):
        with open(path, "w", newline="") as f:
            csv.writer(f).writerows(keep)


def train(config, device=None, num_updates=None, output_dir=None, actor_critic=None, log=print, max_envs_per_pass=None,
          keep_hidden_history=False, tf32_update=False, bf16x3_update=False, native_update=False):
    rank, world = _rank_world()
    device = torch.device(device if device is not None else "cuda:0")
    deterministic = bool(getattr(config.training, "cuda_deterministic", False))
    N, T, H = int(config.training.num_processes), int(config.ppo.num_steps), int(config.sim.human_num)
    resume = _resume_source(config, N, world, rank, deterministic)        # refused here, before any GPU work
    save_state = bool(getattr(config.training, "save_train_state", False))
    state_keys = train_state.run_keys(config, N, world, deterministic) if save_state else None
    torch.manual_seed(config.env.seed + rank)
    torch.cuda.manual_seed_all(config.env.seed + rank)
    if deterministic:
        torch.backends.cudnn.benchmark = False
        torch.backends.cudnn.deterministic = True
    envs = CrowdVecEnv(config, N, device, seed=config.env.seed, phase="train", env_id_offset=rank * N, nenv=N * world)
    if actor_critic is None:
        actor_critic = Policy(envs.observation_space.spaces, envs.action_space, base=config.robot.policy, base_kwargs=config)
    actor_critic.to(device)
    if resume is not None and resume[0] == "weights":
        actor_critic.load_state_dict(resume[1])
        actor_critic.invalidate_weights()
    if world > 1:                         # same initial weights everywhere
        with torch.no_grad():             # in place on the parameter itself: bumps its version, so packed copies are refreshed
            for p in actor_critic.parameters():
                dist.broadcast(p, src=0)
        actor_critic.invalidate_weights()
    rollouts = SRNNRolloutStorage(T, N, envs.observation_space.spaces, envs.action_space, config.SRNN.human_node_rnn_size,
                                  config.SRNN.human_human_edge_rnn_size, "GRU", device=device,
                                  keep_hidden_history=keep_hidden_history)
    agent = PPO(actor_critic, config.ppo.clip_param, config.ppo.epoch, config.ppo.num_mini_batch, config.ppo.value_loss_coef,
                config.ppo.entropy_coef, lr=config.training.lr, eps=config.training.eps,
                max_grad_norm=config.training.max_grad_norm, max_envs_per_pass=max_envs_per_pass, tf32=tf32_update, bf16x3=bf16x3_update,
                native=native_update, deterministic=deterministic)
    obs = envs.reset()
    for k in rollouts.obs:
        rollouts.obs[k][0].copy_(obs[k])
    first = 0
    if resume is not None and resume[0] == "state":
        train_state.restore(resume[1], resume[2], actor_critic, agent.optimizer, envs.engine, rollouts, device)
        first = resume[1]["update"] + 1
    # num_updates counts from the start of the run: a resumed run goes on with update `first` up to the same end
    total_updates = int(config.training.num_env_steps) // T // (N * world)
    if num_updates is None:
        num_updates = total_updates
    out_dir = output_dir if output_dir is not None else config.training.output_dir
    file_log = tboard = None
    if rank == 0 and out_dir:
        os.makedirs(os.path.join(out_dir, "checkpoints"), exist_ok=True)
        file_log = write_run_artefacts(config, out_dir)
        tboard = _tensorboard_writer(out_dir)
        if first:
            _drop_progress_after(os.path.join(out_dir, "progress.csv"), first - 1)
    # device-side episode statistics: [success, collision, timeout, episodes, return sum], reduced ONCE per update from the
    # per-step event / done / episode-return records (three small copies per step instead of ~20 reduction launches)
    stats = torch.zeros(5, dtype=torch.float64, device=device)
    ev_rec = torch.zeros(T, N, dtype=torch.int32, device=device)
    done_rec = torch.zeros(T, N, dtype=torch.bool, device=device)
    ret_rec = torch.zeros(T, N, dtype=torch.float32, device=device)
    history = []
    start = time.time()
    for j in range(first, num_updates):
        if config.training.use_linear_lr_decay:
            update_linear_schedule(agent.optimizer, j, max(total_updates, num_updates), config.training.lr)
        stats.zero_()
        for step in range(T):
            value, action, log_prob, hx = actor_critic.act(rollouts.obs_at(step), dict(rollouts.hidden_at(step)),
                                                           rollouts.masks[step])
            obs, reward, done, buf = envs.step_device(action)
            ev_rec[step].copy_(buf.event.view(N))
            done_rec[step].copy_(done.view(N))
            ret_rec[step].copy_(buf.episode_return.view(N))
            rollouts.insert(obs, hx, action, log_prob, value, reward, buf.not_done, None)     # masks = 1 - done
        d = done_rec.to(torch.float64)
        stats.copy_(torch.stack([((ev_rec == abi.EV_REACH_GOAL) & done_rec).sum().double(),
                                 ((ev_rec == abi.EV_COLLISION) & done_rec).sum().double(),
                                 ((ev_rec == abi.EV_TIMEOUT) & done_rec).sum().double(), d.sum(),
                                 (ret_rec.to(torch.float64) * d).sum()]))
        next_value = actor_critic.get_value(rollouts.obs_at(-1), dict(rollouts.hidden_at(-1)), rollouts.masks[-1]).detach()
        rollouts.compute_returns(next_value, config.ppo.use_gae, config.reward.gamma, config.ppo.gae_lambda,
                                 config.training.use_proper_time_limits)
        value_loss, action_loss, entropy = agent.update(rollouts)
        rollouts.after_update()
        if world > 1:
            dist.all_reduce(stats)
        s = stats.tolist()
        total_steps = (j + 1) * N * world * T
        fps = int((total_steps - first * N * world * T) / (time.time() - start))       # steps of this process only
        row = {"misc/nupdates": j, "misc/total_timesteps": total_steps, "fps": fps,
               "eprewmean": s[4] / s[3] if s[3] else float("nan"), "loss/policy_entropy": entropy,
               "loss/policy_loss": action_loss, "loss/value_loss": value_loss,
               "success": s[0] / s[3] if s[3] else float("nan"), "collision": s[1] / s[3] if s[3] else float("nan"),
               "timeout": s[2] / s[3] if s[3] else float("nan"), "episodes": int(s[3])}
        history.append(row)
        if rank == 0 and out_dir:
            if j % config.training.save_interval == 0 or j == num_updates - 1:
                torch.save(actor_critic.state_dict(), os.path.join(out_dir, "checkpoints", "%.5i" % j + ".pt"))
            if j % config.training.log_interval == 0:
                path = os.path.join(out_dir, "progress.csv")
                fresh = not os.path.exists(path) or j == 0
                with open(path, "w" if fresh else "a", newline="") as f:
                    w = csv.DictWriter(f, fieldnames=list(row)[:7], extrasaction="ignore")
                    if fresh:
                        w.writeheader()
                    w.writerow(row)
        if save_state and out_dir and (j % config.training.save_interval == 0 or j == num_updates - 1):
            train_state.save(os.path.join(out_dir, "checkpoints"), j, total_steps, state_keys, actor_critic, agent.optimizer,
                             envs.engine, rollouts, device, rank, world)
        if rank == 0 and j % config.training.log_interval == 0:
            msg = ("Updates %d, num timesteps %d, FPS %d, episodes %d: mean reward %.3f, success %.3f, collision %.3f, timeout %.3f, "
                   "entropy %.4f, value loss %.4f, policy loss %.5f" % (j, total_steps, row["fps"], row["episodes"], row["eprewmean"],
                                                                         row["success"], row["collision"], row["timeout"], entropy,
                                                                         value_loss, action_loss))
            if log is not None:
                log(msg)
            if file_log is not None:
                file_log.info(msg)
            if tboard is not None:          # train.py:376-386
                tboard.add_scalar("mean_reward", row["eprewmean"], total_steps)
                tboard.add_scalar("policy_entropy (dist_entropy)", entropy, total_steps)
                tboard.add_scalar("policy_loss (action_loss)", action_loss, total_steps)
                tboard.add_scalar("value_loss", value_loss, total_steps)
    if file_log is not None:
        for h in list(file_log.handlers):
            h.close()
            file_log.removeHandler(h)
    if tboard is not None:
        tboard.close()
    envs.close()
    return actor_critic, history


def main(argv=None):
    """`python -m crowdnav_dsrnn_b200.train [--output_dir DIR] [--num_updates K] [--envs N] [--humans H] [--native]
    [--deterministic] [--save-state] [--resume PATH]`:
    the reference's `python train.py` on the batched backend (its settings come from the config file; here the ones that
    matter for a batch of thousands of envs can be given on the command line)."""
    import argparse

    from .config import Config

    ap = argparse.ArgumentParser("crowdnav_dsrnn_b200.train")
    ap.add_argument("--output_dir", default=None)
    ap.add_argument("--num_updates", type=int, default=None)
    ap.add_argument("--envs", type=int, default=None, help="training.num_processes (envs per GPU)")
    ap.add_argument("--humans", type=int, default=None)
    ap.add_argument("--kinematics", default="holonomic", choices=["holonomic", "unicycle"])
    ap.add_argument("--envs_per_pass", type=int, default=4096)
    ap.add_argument("--native", action="store_true", help="PPO update on the library's own tensor-core kernels")
    ap.add_argument("--deterministic", action="store_true",
                    help="training.cuda_deterministic: the same seed gives the same checkpoints (ordered reductions in the update)")
    ap.add_argument("--save-state", dest="save_state", action="store_true",
                    help="training.save_train_state: write training-state files (%%.5i.state.pt) next to the checkpoints")
    ap.add_argument("--resume", default=None, metavar="PATH",
                    help="training.resume from training.load_path = PATH: a training-state file continues that run, a "
                         "state_dict starts a fresh run from its weights")
    args = ap.parse_args(argv)
    cfg = Config(kinematics=args.kinematics, human_num=args.humans)
    if args.deterministic:
        cfg.training.cuda_deterministic = True
    if args.save_state:
        cfg.training.save_train_state = True
    if args.resume:
        cfg.training.resume = True
        cfg.training.load_path = args.resume
    if args.envs:
        cfg.training.num_processes = args.envs
    if args.output_dir:
        cfg.training.output_dir = args.output_dir
    if dist.is_available() and "RANK" in os.environ and not dist.is_initialized():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    train(cfg, device, num_updates=args.num_updates, max_envs_per_pass=args.envs_per_pass, native_update=args.native)
    return 0


if __name__ == "__main__":
    sys.exit(main())
