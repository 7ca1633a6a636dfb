"""CPU: the C oracle (oracle/crowd_oracle.c) against the golden vectors produced by the reference's own
CrowdSimDict.step (oracle/gen_golden.py), at the north_star tolerances (flags bit-exact); the DS-RNN restatement
(oracle/dsrnn_oracle.py) against the reference's own Policy.act on the stored inputs (oracle/gen_golden_dsrnn.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import crowd_oracle, dsrnn_oracle
from helpers import DSRNN_CASES, GOLDEN, STEP_CASES, check_against_reference, load_step_case


def test_golden_fixtures_present():
    assert {"c1_holonomic_h5", "c2_unicycle_h10", "c3_fov_h20", "c4_social_h5", "c4_sidepref_h1"} <= set(STEP_CASES)


@pytest.mark.parametrize("name", STEP_CASES)
def test_oracle_step_matches_reference(name):
    d, _, cfg, n = load_step_case(name)
    st = crowd_oracle.OracleState(n, cfg.human_num)
    for f in ("robot", "humans", "belief", "extras", "counters"):
        getattr(st, f)[...] = d["in_" + f]
    out = crowd_oracle.step(cfg, st, d["in_action"], auto_reset=False)
    check_against_reference(d, cfg, out.as_dict(), st.as_dict(), where=name)


@pytest.mark.parametrize("name", ["c1_holonomic_h5", "c3_fov_h20"])
def test_oracle_threads_agree(name):
    d, _, cfg, n = load_step_case(name)
    outs = []
    for threads in (1, 4):
        st = crowd_oracle.OracleState(n, cfg.human_num)
        for f in ("robot", "humans", "belief", "extras", "counters"):
            getattr(st, f)[...] = d["in_" + f]
        o = crowd_oracle.step(cfg, st, d["in_action"], auto_reset=True, n_threads=threads)
        outs.append((o.as_dict(), st.as_dict()))
    for a, b in zip(outs[0], outs[1]):
        for k in a:
            assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("case", DSRNN_CASES)
def test_dsrnn_restatement_matches_reference_policy(case):
    """The torch restatement smoke() and the GPU forward tests compare with, against the reference Policy (shipped checkpoints)."""
    d = np.load(os.path.join(GOLDEN, "dsrnn_%s.npz" % case))
    w = np.load(os.path.join(GOLDEN, "weights_%s.npz" % case.rsplit("_h", 1)[0]))
    t = lambda k: torch.from_numpy(d[k])
    mine = dsrnn_oracle.forward({k: torch.from_numpy(w[k]) for k in w.files}, t("robot_node"), t("temporal_edges"),
                                t("spatial_edges"), t("h_node"), t("h_edge"), t("masks"))
    for k, tol in (("value", 1e-4), ("action_mean", 1e-4), ("actor_features", 1e-4), ("h_node", 1e-5), ("h_edge", 1e-5)):
        assert float((mine[k] - t("ref_" + k).reshape(mine[k].shape)).abs().max()) <= tol, k
