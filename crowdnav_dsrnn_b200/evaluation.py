"""Batched evaluator (SURVEY.md 8(f) N2): the test loop of pytorchBaselines/evaluation.py:96-330 with the
`env.test_size` episodes played as ONE batch on the GPU instead of one after the other in a single env.

Env k of the batch plays what would have been the k-th test episode of the reference's single env: its
`scenario_counter` starts at k (sequential scenarios under test.social_metrics, crowd_sim_dict.py:114-122) and its
`case_counter` at k (seed = 1000 + k + env.seed, crowd_sim_dict.py:147-154).  The reference carries
`last_acceleration` from one episode into the next (it is initialised in `configure` only, crowd_sim.py:208), which
shows up in the first jerk sample (SM4) of every episode; to reproduce that, every env first plays `warmup_episodes`
unscored episodes (env k starts at counter k - warmup) and the NEXT one is scored.  The rollout stops when every env
has finished its scored episode.  Per-step social metrics (SM1-SM6, evaluation.py:155-190) are accumulated on the
device from the step-info columns.

With a model-based robot (robot.policy = 'orca' / 'social_force') the robot acts by itself inside the vectorised env's
step: `actor_critic` is None and no forward runs, everything else is the same.
"""
import math

import numpy as np
import torch

from . import abi
from .envs import CrowdVecEnv


@torch.no_grad()
def evaluate_batched(actor_critic, config, device, episodes=None, seed=None, deterministic=True, warmup_episodes=1,
                     return_episodes=False):
    robot_policy = abi.robot_policy_of(config)
    if robot_policy is not None and actor_critic is not None:
        raise ValueError("robot.policy=%r acts by itself: evaluate it with actor_critic=None" % (config.robot.policy,))
    if robot_policy is None and actor_critic is None:
        raise ValueError("robot.policy='srnn' needs the actor_critic that drives it")
    n = int(config.env.test_size if episodes is None else episodes)
    device = torch.device(device)
    venv = CrowdVecEnv(config, n, device, seed=config.env.seed if seed is None else seed, phase="test", nenv=1)
    eng = venv.engine
    H = config.sim.human_num
    st = eng.get_state()
    W = int(warmup_episodes)
    size = max(1, int(eng.cfg.case_size))
    ks = torch.arange(n, dtype=torch.int64, device=device) - W
    st["counters"][:, 1] = (ks % 4 + 4).to(torch.int32)          # same residue mod 4, never negative
    st["counters"][:, 2] = (ks % size).to(torch.int32)
    eng.set_state(counters=st["counters"])
    obs = eng.reset().obs()
    hx = None if actor_critic is None else {"human_node_rnn": torch.zeros(n, 1, 128, device=device),
                                            "human_human_edge_rnn": torch.zeros(n, H + 1, 256, device=device)}
    action = None
    masks = torch.zeros(n, 1, device=device)
    finished = torch.zeros(n, dtype=torch.bool, device=device)
    ep_idx = torch.zeros(n, dtype=torch.int32, device=device)      # episodes completed so far by each env
    event = torch.zeros(n, dtype=torch.int32, device=device)
    scenario = torch.zeros(n, dtype=torch.int32, device=device)
    length = torch.zeros(n, dtype=torch.int32, device=device)
    ret = torch.zeros(n, device=device)
    col = abi.INFO_COLUMNS
    acc = {k: torch.zeros(n, device=device) for k in ("personal_violation", "path_violation", "aggregate_nav_time",
                                                       "jerk_cost", "speed_violation", "side_left", "side_right")}
    path_len = torch.zeros(n, device=device)
    chc = torch.zeros(n, device=device)                            # cumulative heading change (evaluation.py:145-150)
    disc_ret = torch.zeros(n, dtype=torch.float64, device=device)  # sum gamma^(t dt v_pref) r_t (evaluation.py:205-208)
    t_in_ep = torch.zeros(n, dtype=torch.float64, device=device)
    log_gamma_step = math.log(0.99) * float(config.env.time_step) * float(config.robot.v_pref)
    last_pos = obs["robot_node"][:, 0, 0:2].clone()
    last_angle = torch.atan2(obs["temporal_edges"][:, 0, 1], obs["temporal_edges"][:, 0, 0])
    for _ in range((W + 1) * (int(eng.cfg.timeout_step) + 2)):
        if actor_critic is not None:
            _, action, _, hx = actor_critic.act(obs, hx, masks, deterministic=deterministic)
        obs, _, done, buf = venv.step_device(action)
        live = ep_idx == W                                          # currently playing the scored episode
        for k in acc:
            acc[k] += torch.where(live, buf.info[:, col[k]], torch.zeros_like(ret))
        pos = obs["robot_node"][:, 0, 0:2]
        path_len += torch.where(live, (pos - last_pos).norm(dim=-1), torch.zeros_like(ret))   # evaluation.py:134-143
        last_pos = pos.clone()
        angle = torch.atan2(obs["temporal_edges"][:, 0, 1], obs["temporal_edges"][:, 0, 0])
        chc += torch.where(live, (angle - last_angle).abs(), torch.zeros_like(ret))
        last_angle = angle
        disc_ret += torch.where(live, torch.exp(t_in_ep * log_gamma_step) * buf.reward.double(), torch.zeros_like(disc_ret))
        t_in_ep = torch.where(done.bool(), torch.zeros_like(t_in_ep), t_in_ep + 1.0)
        first = live & done.bool()
        ep_idx += done.to(torch.int32)
        event = torch.where(first, buf.event, event)
        scenario = torch.where(first, buf.scenario, scenario)
        length = torch.where(first, buf.episode_length, length)
        ret = torch.where(first, buf.episode_return, ret)
        finished |= first
        masks = buf.not_done                                        # 1 - done, written by the step kernel
        if bool(finished.all()):
            break
    venv.close()
    ev = event.cpu()
    scn = scenario.cpu()
    steps = length.cpu().float()
    dt = float(config.env.time_step)
    out = {
        "episodes": n,
        "success": float((ev == abi.EV_REACH_GOAL).float().mean()),
        "collision": float((ev == abi.EV_COLLISION).float().mean()),
        "timeout": float((ev == abi.EV_TIMEOUT).float().mean()),
        "unfinished": int((~finished).sum()),
        "mean_steps": float(steps.mean()),
        "mean_steps_success": float(steps[ev == abi.EV_REACH_GOAL].mean()) if bool((ev == abi.EV_REACH_GOAL).any()) else float("nan"),
        "mean_nav_time_success": float(steps[ev == abi.EV_REACH_GOAL].mean()) * dt if bool((ev == abi.EV_REACH_GOAL).any()) else float("nan"),
        "mean_return": float(ret.mean()),
        "mean_path_length": float(path_len.mean()),
        "per_scenario": {},
    }
    for k, v in acc.items():                     # per-episode sums of the per-step values (evaluation.py:155-190 multiplies
        out["mean_" + k + "_per_episode"] = float(v.mean())   # the violation counts by time_step when it logs them)
        out["std_" + k + "_per_episode"] = float(v.std())
    # side preference: an episode is labelled with the side seen most often (evaluation.py:199-210)
    out["side_left_episodes"] = float((acc["side_left"] > acc["side_right"]).float().mean())
    out["side_right_episodes"] = float((acc["side_right"] > acc["side_left"]).float().mean())
    if return_episodes:
        out["episode_detail"] = {"event": ev.numpy(), "scenario": scn.numpy(), "steps": length.cpu().numpy(),
                                 "return": ret.cpu().numpy(), "discounted_return": disc_ret.cpu().numpy(),
                                 "path_length": path_len.cpu().numpy(), "chc": chc.cpu().numpy(),
                                 **{k: v.cpu().numpy() for k, v in acc.items()}}
    for s in sorted(set(scn.tolist())):
        sel = scn == s
        out["per_scenario"][abi.SCENARIOS[s]] = {
            "episodes": int(sel.sum()), "success": float((ev[sel] == abi.EV_REACH_GOAL).float().mean()),
            "collision": float((ev[sel] == abi.EV_COLLISION).float().mean()),
            "timeout": float((ev[sel] == abi.EV_TIMEOUT).float().mean())}
    return out


def _log_metric(logging, name, sample):
    """Metrics.add_metric + log_metrics of pytorchBaselines/metrics.py:10-45 (mean, std, 90 % t-interval)."""
    from scipy import stats

    sample = np.asarray(sample, dtype=np.float64)
    mean, std = (float(np.mean(sample)), float(np.std(sample))) if sample.size else (float("nan"), float("nan"))
    if sample.size > 1:
        lo, hi = stats.t.interval(0.9, sample.size - 1, mean, stats.sem(sample))
    else:
        lo, hi = float("nan"), float("nan")
    logging.info("")
    logging.info(f"{name} ======")
    logging.info(f"MEAN: {mean:.4f}")
    logging.info(f"STD DEV: {std:.4f}")
    logging.info(f"CI: [{lo:.4f},{hi:.4f}]")


def evaluate(actor_critic, ob_rms, eval_envs, num_processes, device, config, logging, visualize=False, recurrent_type="GRU"):
    """Drop-in for pytorchBaselines/evaluation.py:14-334 (test.py:204-214): same signature, same log lines, same return
    triple -- but the `env.test_size` episodes are played as ONE batch on the GPU (`evaluate_batched`), not one after the
    other in `eval_envs` (which is only closed, as the reference does at the end).  Episode k of the reference is env k of
    the batch.  The returned dicts hold one `[episode total]` list per episode (the per-step traces that
    test.py --study_scenario plots are not kept on the host); `dist_to_goal` is left empty.  A model-based robot
    (robot.policy = 'orca' / 'social_force') is evaluated with actor_critic=None."""
    if visualize:
        raise NotImplementedError("rendering is out of scope (SURVEY section 2 row 2)")
    if recurrent_type != "GRU":
        raise NotImplementedError("only GRU cells are on the DS-RNN path")
    res = evaluate_batched(actor_critic, config, device, return_episodes=True)
    d = res["episode_detail"]
    n, dt = res["episodes"], float(config.env.time_step)
    ev, scn = d["event"], d["scenario"]
    names = {abi.EV_REACH_GOAL: "success", abi.EV_COLLISION: "collision", abi.EV_TIMEOUT: "timeout"}
    cases = {k: [int(i) for i in np.nonzero(ev == e)[0]] for e, k in names.items()}
    raw = {k: [[float(d["return"][i])] for i in cases[k]] for k in names.values()}
    disc = {k: [[float(d["discounted_return"][i])] for i in cases[k]] for k in names.values()}
    d2g = {k: [] for k in names.values()}
    scenarios = sorted(set(config.sim.train_val_sim) | set(config.sim.test_sim))
    num_events = {k: dict(total=len(cases[k]), **{s: 0 for s in scenarios}) for k in names.values()}
    for k in names.values():
        for i in cases[k]:
            num_events[k][abi.SCENARIOS[int(scn[i])]] = num_events[k].get(abi.SCENARIOS[int(scn[i])], 0) + 1
    ok = np.asarray(cases["success"], dtype=np.int64)
    logging.info("TEST")
    # evaluation.py:156 tests a dict against Danger, so the reference never records a min distance: 0 time in danger, nan
    logging.info(f"Total time in danger: {0.0:.4f}, average min distance in danger: {float('nan'):.4f}")
    logging.info(f"success rate: {len(cases['success']) / n:.3f}")
    logging.info(f"collision rate: {len(cases['collision']) / n:.3f}")
    logging.info(f"timeout rate: {len(cases['timeout']) / n:.3f}")
    logging.info("Success cases: " + " ".join(str(x) for x in cases["success"]))
    logging.info("Collision cases: " + " ".join(str(x) for x in cases["collision"]))
    logging.info("Timeout cases: " + " ".join(str(x) for x in cases["timeout"]))
    logging.info("")
    logging.info("SCENARIO BREAKDOWN: ")
    for k in num_events:                                    # helper.py:88-101
        logging.info("")
        logging.info(f"{k.upper()} CASES: ")
        for scenario, count in num_events[k].items():
            logging.info(f"{scenario}: {count}")
    # the reference reads global_time before the terminal step (evaluation.py:128-129): (steps - 1) * dt
    _log_metric(logging, "navigation time", (d["steps"][ok] - 1) * dt)
    _log_metric(logging, "path length", d["path_length"][ok])
    order = [i for k in ("success", "collision", "timeout") for i in cases[k]]
    _log_metric(logging, "discounted reward", d["discounted_return"][order])
    _log_metric(logging, "non-discounted rewards", d["return"][order])
    _log_metric(logging, "cumulative heading change", d["chc"][ok])
    if config.test.social_metrics:                          # appended for successful episodes only (evaluation.py:213-228)
        _log_metric(logging, "SM1 - personal space violation", d["personal_violation"][ok] * dt)
        _log_metric(logging, "SM2 - path violation", d["path_violation"][ok] * dt)
        _log_metric(logging, "SM3 - aggregate time", d["aggregate_nav_time"][ok] * dt)
        _log_metric(logging, "SM4 - jerk cost", d["jerk_cost"][ok])
        _log_metric(logging, "SM5 - speed violation", d["speed_violation"][ok] * dt)
    if config.test.side_preference:
        scenario = config.sim.test_sim[0]
        left = float(np.sum(d["side_left"][ok] > d["side_right"][ok])) / n
        right = float(np.sum(d["side_left"][ok] < d["side_right"][ok])) / n
        logging.info("")
        logging.info(f"Side Preference - {scenario} ======")
        logging.info(f"Left % = {100 * left:.3f}%")
        logging.info(f"Right % = {100 * right:.3f}%")
    if eval_envs is not None and hasattr(eval_envs, "close"):
        eval_envs.close()
    return raw, disc, d2g
