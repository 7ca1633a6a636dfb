import os, sys, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import DSRNN_CASES, GOLDEN
from test_gpu_dsrnn import _policy, _rel_err
for prec in ("bf16x3", "fp16", "bf16"):
    worst = {}
    for case in DSRNN_CASES:
        ckpt, h = case.rsplit("_h", 1); H = int(h)
        d = np.load(os.path.join(GOLDEN, "dsrnn_%s.npz" % case)); w = np.load(os.path.join(GOLDEN, "weights_%s.npz" % ckpt))
        policy, _ = _policy(H, {k: w[k] for k in w.files}); policy.precision = prec
        t = lambda k: torch.from_numpy(d[k]).cuda()
        obs = {"robot_node": t("robot_node"), "temporal_edges": t("temporal_edges"), "spatial_edges": t("spatial_edges")}
        value, mean, feat, hn, he = policy.cuda_forward(obs, {"human_node_rnn": t("h_node"), "human_human_edge_rnn": t("h_edge")}, t("masks"))
        for k, got in (("value", value), ("action_mean", mean), ("h_node", hn), ("h_edge", he)):
            worst[k] = max(worst.get(k, 0), _rel_err(got.cpu().numpy(), d["ref_" + k]))
    print(prec, {k: "%.2e" % v for k, v in worst.items()})
