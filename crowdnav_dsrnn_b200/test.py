"""`python -m crowdnav_dsrnn_b200.test`: the reference's test.py (test.py:25-214) on the batched backend -- same
command-line flags, same model-directory layout (`<model_dir>/configs/train_config.py`, `<model_dir>/checkpoints/*.pt`),
same log file name (`<model_dir>/test/model_<ckpt>_test_<name>_.log`, test.py:103-128) and the log lines of
pytorchBaselines/evaluation.py:283-330; the `env.test_size` test episodes are played as one batch on the GPU.

--robot_policy orca / social_force evaluates a model-based robot instead of a checkpoint: config.robot.policy is
overridden, no checkpoint is loaded, `--model_dir` still supplies the config and the log directory, and the log file is
named as if the policy were the checkpoint (`model_orca_test_<name>_.log`).

--viz / --study_scenario need the renderer / per-step traces, which are out of scope (SURVEY section 2 row 2)."""
import argparse
import importlib
import logging
import os
import sys
from pathlib import Path

import numpy as np
import torch

from .envs import make_vec_envs
from .evaluation import evaluate
from .model import Policy


def _load_config(model_dir, default_config=True):
    """test.py:84-98: the Config class saved next to the model, else this package's restatement of the defaults."""
    if default_config:
        mod = model_dir.rstrip("/").replace("/", ".") + ".configs.train_config"
        try:
            return getattr(importlib.import_module(mod), "Config")()
        except Exception:  # noqa: BLE001 - same fall-back as the reference's bare except
            print("Failed to get train_config from %s, loading default CrowdNav config" % model_dir)
    from .config import Config

    return Config()


def log_file_name(test_model, test_name):
    """test.py:108-118."""
    f_name = ""
    if test_model:
        f_name += "model_" + str(Path(test_model).with_suffix("")) + "#"
    if test_name:
        f_name += "test_" + test_name + "#"
    return (f_name + ".log").replace("#", "_")


def main(argv=None):
    ap = argparse.ArgumentParser("Parser for test.py", add_help=True)
    ap.add_argument("--model_dir", type=str, default="data/example_model")
    ap.add_argument("--viz", action="store_true")
    ap.add_argument("--test_case", type=int, default=-1)
    ap.add_argument("--test_model", type=str, default=None)
    ap.add_argument("--test_name", type=str, default="test")
    ap.add_argument("--default_config", type=bool, default=True)
    ap.add_argument("--num_threads", type=int, default=1)
    ap.add_argument("--study_scenario", action="store_true")
    ap.add_argument("--robot_policy", type=str, default=None, choices=["orca", "social_force"],
                    help="evaluate a model-based robot instead of a checkpoint")
    args = ap.parse_args(argv)
    if args.viz or args.study_scenario:
        raise NotImplementedError("--viz / --study_scenario need the renderer (out of scope, SURVEY section 2 row 2)")
    model_dir = args.model_dir.rstrip("/")
    if os.getcwd() not in sys.path:
        sys.path.insert(0, os.getcwd())
    if args.robot_policy is not None:
        args.test_model = args.robot_policy
    elif args.test_model is None:                # test.py:61-81: newest checkpoint of the run
        args.test_model = sorted(os.listdir(os.path.join(model_dir, "checkpoints")), reverse=True)[0]
    config = _load_config(model_dir, args.default_config)
    if args.robot_policy is not None:
        config.robot.policy = args.robot_policy
    log_dir = Path.cwd() / model_dir / "test"
    log_dir.mkdir(parents=True, exist_ok=True)
    log_file = str(log_dir / log_file_name(args.test_model, args.test_name))
    logger = logging.getLogger("crowdnav_dsrnn_b200.test")
    logger.setLevel(logging.INFO)
    logger.propagate = False
    for h in list(logger.handlers):
        logger.removeHandler(h)
    fmt = logging.Formatter("%(asctime)s, %(levelname)s: %(message)s", datefmt="%Y-%m-%d %H:%M:%S")
    for h in (logging.StreamHandler(sys.stdout), logging.FileHandler(log_file, mode="w")):
        h.setFormatter(fmt)
        logger.addHandler(h)
    if args.test_case != -1:
        config.env.test_size = 1
    logger.info("Test Cases: " + ("all" if args.test_case == -1 else str(args.test_case)))
    logger.info("robot FOV %f", config.robot.FOV * np.pi)
    logger.info("humans FOV %f", config.humans.FOV * np.pi)
    torch.manual_seed(config.env.seed)
    torch.cuda.manual_seed_all(config.env.seed)
    torch.set_num_threads(args.num_threads)
    device = torch.device("cuda:0")
    if args.robot_policy is not None:
        logger.info("Using robot policy %s" % args.robot_policy)
    else:
        load_path = str(Path.cwd() / model_dir / "checkpoints" / args.test_model)
        logger.info("Using model %s" % load_path)
    envs = make_vec_envs(config.env.env_name, config.env.seed, 1, config.reward.gamma, None, device, allow_early_resets=True,
                         config=config, test_case=args.test_case)
    actor_critic = None
    if args.robot_policy is None:
        actor_critic = Policy(envs.observation_space.spaces, envs.action_space, base_kwargs=config, base=config.robot.policy)
        actor_critic.load_state_dict(torch.load(load_path, map_location=device))
        actor_critic.base.nenv = 1
        actor_critic.to(device)
    evaluate(actor_critic=actor_critic, ob_rms=False, eval_envs=envs, num_processes=1, device=device, config=config,
             logging=logger, visualize=False, recurrent_type="GRU")
    for h in list(logger.handlers):
        h.close()
        logger.removeHandler(h)
    return 0


if __name__ == "__main__":
    sys.exit(main())
