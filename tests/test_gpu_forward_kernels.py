"""GPU: the rollout forward cn_dsrnn_forward stage by stage against float64 references, in all four precision modes --
the edge GRUs (edge_gru_tc_kernel, rollout instantiation, or edge_gru_simt_kernel in fp32 mode), the folded query
projection (linear_tc_kernel / linear_simt_kernel), the online-softmax attention_kernel and the node / heads stage
(node_heads_tc_kernel, or the fp32 chain node_encode_kernel -> linear_simt_kernel -> node_gru_gate_kernel -> heads_kernel)
-- at the benchmark shapes, with what the forward must not write or read, the resident edge image of the graphed rollout
and the re-packing of the weight images after an update.

Every reference is plain torch in float64 on the GPU, and each stage's reference is fed the kernel's own output of the
stage before, so an error is charged to the stage that made it.  Each check prints its worst error next to its tolerance
(run with -s to see the margins)."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from crowdnav_dsrnn_b200 import Config, _lib, abi, native
from crowdnav_dsrnn_b200.model import Policy
from crowdnav_dsrnn_b200.spaces import crowd_spaces
from oracle import dsrnn_oracle
from helpers import GOLDEN

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
F64 = torch.float64
BF16 = torch.bfloat16
MODES = ("fp32", "bf16x3", "fp16", "bf16")     # from the most to the least accurate
P = native._ptr


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _check(name, got, want, tol, floor=1.0):
    """max |got - want| <= tol * max(floor, max |want|); a NaN in `got` fails."""
    scale = max(floor, want.abs().max().item())
    err = (got.double() - want).abs().max().item()
    print("%-64s err %.3e of scale %.3e = %.2e (tol %.1e)" % (name, err, scale, err / scale, tol))
    assert err <= tol * scale, (name, err, scale)


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _same_bits(a, b):
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _split(x):
    """bf16(x), bf16(x - bf16(x)): the split image the bf16x3 kernels read and write."""
    hi = x.bfloat16()
    return hi, (x - hi.float()).bfloat16()


def _ws_views(ws, N):
    """qt [N, 256] and cat = [o_t | c] [N, 512], both fp32, inside the forward's workspace: carve_ws in
    csrc/dsrnn_forward.cu places qt at byte 0 and cat right after it (N * 1024 bytes is a multiple of its 256-byte
    alignment)."""
    f = ws.view(torch.float32)
    return f[:N * 256].view(N, 256), f[N * 256:N * 768].view(N, 512)


# ------------------------------------------------------------------------------------------------ weights and inputs
def _make_policy(sd):
    obs_space, act_space = crowd_spaces(5)        # no weight depends on human_num: one handle serves every H
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        policy = Policy(obs_space.spaces, act_space, base="srnn", base_kwargs=Config(human_num=5))
    policy.load_state_dict({k: torch.as_tensor(v) for k, v in sd.items()})
    return policy.to(DEV)


def _checkpoint(name):
    w = np.load(os.path.join(GOLDEN, "weights_%s.npz" % name))
    return {k: w[k] for k in w.files}


ATT_T, ATT_S = "base.attn.temporal_edge_layer.0.", "base.attn.spatial_edge_layer.0."


def _large_logit_state_dict(seed, logit=300.0):
    """Random weights whose attention layers are scaled so that the rollout softmax sees scores q.k_i * H / 8 of about
    +-`logit` at H = 20 on synthetic inputs (exp(300) overflows fp32: the online softmax must subtract its running max).
    Calibrated on the float64 edge outputs of a seeded probe batch."""
    sd = dsrnn_oracle.random_state_dict(seed=seed)
    p = {k: v.double() for k, v in sd.items()}
    g = torch.Generator().manual_seed(seed)
    n, H = 256, 20
    probe = {"temporal_edges": torch.randn(n, 1, 2, generator=g), "spatial_edges": torch.randn(n, H, 2, generator=g) * 4,
             "h_edge": torch.randn(n, H + 1, 256, generator=g) * 0.5, "masks": torch.ones(n, 1)}
    o = _edge_reference(p, probe)
    q = _lin(p, ATT_T, o[:, 0])
    s = torch.einsum("bd,bhd->bh", q, o[:, 1:] @ p[ATT_S + "weight"].t()) * (H / 8.0)
    f = math.sqrt(logit / s.abs().max().item())
    for k in (ATT_T + "weight", ATT_T + "bias", ATT_S + "weight"):
        sd[k] = sd[k] * f
    return sd


@pytest.fixture(scope="module")
def policies():
    """The two shipped checkpoints, a random policy whose edge-GRU weights are scaled x4 (the gates cover their whole
    range instead of sitting near 0.5) and a random policy with rollout softmax logits of about +-300."""
    edge = dsrnn_oracle.random_state_dict(seed=2024)
    for k in edge:
        if "EdgeRNN" in k and ".gru." in k:
            edge[k] = edge[k] * 4.0
    out = {"holonomic_27776": _make_policy(_checkpoint("holonomic_27776")),
           "unicycle_55554": _make_policy(_checkpoint("unicycle_55554")),
           "edge_x4": _make_policy(edge),
           "logits300": _make_policy(_large_logit_state_dict(seed=7))}
    yield out
    for p in out.values():
        if p._handle is not None:
            p.set_edge_image(None, None)


def _masks(kind, N, seed):
    if kind == "zeros":
        return torch.zeros(N, 1, device=DEV)
    if kind == "ones":
        return torch.ones(N, 1, device=DEV)
    keep = (torch.rand(N, 1, device=DEV, generator=_gen(seed)) > 0.2).float()
    if kind == "mixed":
        return keep
    assert kind == "fractional"        # the ABI takes float masks: 0, 0.5 and values in between
    frac = torch.rand(N, 1, device=DEV, generator=_gen(seed + 1))
    return keep * torch.where(frac < 0.5, torch.full_like(frac, 0.5), frac)


def _synthetic(N, H, masks, seed):
    """The input distribution of test_forward_matches_torch_restatement."""
    g = _gen(seed)
    r = lambda *s: torch.randn(*s, device=DEV, generator=g)
    return {"robot_node": r(N, 1, 7) * 3, "temporal_edges": r(N, 1, 2), "spatial_edges": r(N, H, 2) * 4,
            "h_node": r(N, 1, 128) * 0.5, "h_edge": r(N, H + 1, 256) * 0.5, "masks": _masks(masks, N, seed + 7)}


@pytest.fixture(scope="module")
def realistic(policies):
    """What the network sees in the c3 benchmark: the observation, hidden states and masks after 20 eager act ->
    step_device steps of 16384 envs with robot.FOV 0.5 and 20 humans under the shipped holonomic checkpoint (distances,
    dummy edges of unseen humans, episodes that ended)."""
    from crowdnav_dsrnn_b200.envs import CrowdVecEnv

    cfg = Config(kinematics="holonomic", human_num=20)
    cfg.robot.FOV = 0.5
    N = 16384
    venv = CrowdVecEnv(cfg, N, DEV, seed=5)
    policy = policies["holonomic_27776"]
    obs = venv.reset()
    hx = {"human_node_rnn": torch.zeros(N, 1, 128, device=DEV), "human_human_edge_rnn": torch.zeros(N, 21, 256, device=DEV)}
    masks = torch.zeros(N, 1, device=DEV)
    with torch.random.fork_rng(devices=[DEV]):
        torch.manual_seed(0)
        for _ in range(20):
            _, action, _, hx = policy.act(obs, hx, masks)
            obs, _, _, buf = venv.step_device(action)
            masks = buf.not_done
    inp = {"robot_node": obs["robot_node"], "temporal_edges": obs["temporal_edges"], "spatial_edges": obs["spatial_edges"],
           "h_node": hx["human_node_rnn"], "h_edge": hx["human_human_edge_rnn"], "masks": masks}
    inp = {k: v.clone() for k, v in inp.items()}
    torch.cuda.synchronize()
    venv.close()
    assert 0 < int((inp["masks"] == 0).sum()) < N                 # some episodes ended in the last step
    return inp


# ------------------------------------------------------------------------------------------------ the forward
def _workspace(N, H):
    nbytes = _lib.load().cn_dsrnn_workspace_bytes(N, H)
    return torch.full(((nbytes + 3) // 4,), float("nan"), device=DEV).view(torch.uint8)


def _cuda_forward(policy, inp, mode, ws=None):
    """Policy.cuda_forward with caller-owned outputs and workspace (so that every stage can be read back)."""
    N, H = inp["spatial_edges"].shape[:2]
    ws = _workspace(N, H) if ws is None else ws
    out = {"h_node": torch.empty(N, 1, 128, device=DEV), "h_edge": torch.empty(N, H + 1, 256, device=DEV),
           "value": torch.empty(N, 1, device=DEV), "mean": torch.empty(N, 2, device=DEV)}
    obs = {k: inp[k] for k in ("robot_node", "temporal_edges", "spatial_edges")}
    hx = {"human_node_rnn": inp["h_node"], "human_human_edge_rnn": inp["h_edge"]}
    policy.precision = mode
    try:
        value, mean, feat, hn, he = policy.cuda_forward(obs, hx, inp["masks"], out=out, workspace=ws)
    finally:
        policy.precision = "bf16x3"
    torch.cuda.synchronize()
    return dict(value=value, mean=mean, feat=feat, h_node=hn, h_edge=he), ws


def _abi_forward(policy, inp, mode, out, ws):
    """cn_dsrnn_forward through the C ABI into caller-given outputs (out["feat"] may be None)."""
    N, H = inp["spatial_edges"].shape[:2]
    lib = policy._ensure_handle(DEV)
    io = abi.CnDsrnnIO(P(inp["robot_node"]), P(inp["temporal_edges"]), P(inp["spatial_edges"]), P(inp["h_node"]),
                       P(inp["h_edge"]), P(inp["masks"]), P(out["h_node"]), P(out["h_edge"]), P(out["value"]),
                       P(out["mean"]), P(out["feat"]))
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    _lib.check(lib.cn_dsrnn_forward(policy._handle, N, H, C.byref(io), abi.PRECISIONS[mode], P(ws), ws.numel(), stream),
               "cn_dsrnn_forward")


# ------------------------------------------------------------------------------------------------ float64 references
def _params64(policy):
    return {k: v.detach().double() for k, v in policy.state_dict().items()}


def _lin(p, key, x):
    return x @ p[key + "weight"].t() + p[key + "bias"]


def _gru_step(p, key, x, h):
    """torch.nn.GRU step, gate order r|z|n: h' = n + z (h - n)."""
    gi, gh = _lin_gru(p, key, "ih", x), _lin_gru(p, key, "hh", h)
    n_h = h.shape[1]
    r = torch.sigmoid(gi[:, :n_h] + gh[:, :n_h])
    z = torch.sigmoid(gi[:, n_h:2 * n_h] + gh[:, n_h:2 * n_h])
    n = torch.tanh(gi[:, 2 * n_h:] + r * gh[:, 2 * n_h:])
    return n + z * (h - n)


def _lin_gru(p, key, which, x):
    return x @ p[key + "weight_%s_l0" % which].t() + p[key + "bias_%s_l0" % which]


def _chunks(N, rows_per_env, budget=1 << 19):
    step = max(1, budget // rows_per_env)
    return [(e0, min(N, e0 + step)) for e0 in range(0, N, step)]


def _edge_reference(p, inp):
    """Both edge GRUs for one step: e = ReLU(W_enc x + b), hm = m h, GRU step; [N, H + 1, 256] (row 0 temporal)."""
    N, H = inp["spatial_edges"].shape[:2]
    out = torch.empty(N, H + 1, 256, dtype=F64, device=inp["h_edge"].device)
    for e0, e1 in _chunks(N, H + 1):
        n = e1 - e0
        hm = inp["h_edge"][e0:e1].double() * inp["masks"][e0:e1].double().view(n, 1, 1)
        for pre, x, h, dst in (("temporal", inp["temporal_edges"][e0:e1].reshape(n, 2), hm[:, 0], out[e0:e1, 0]),
                               ("spatial", inp["spatial_edges"][e0:e1].reshape(n * H, 2), hm[:, 1:].reshape(n * H, 256),
                                out[e0:e1, 1:])):
            key = "base.humanhumanEdgeRNN_%s." % pre
            e = torch.relu(_lin(p, key + "encoder_linear.", x.double()))
            dst.copy_(_gru_step(p, key + "gru.", e, h).view(dst.shape))
    return out


def _attention_reference(p, h_edge, qt):
    """From the kernel's own h_edge_out (o_t = row 0, o_i = rows 1..H) and qt: the unfolded query projection
    W_s^T (W_t o_t + b_t), and c = sum_i alpha_i o_i with alpha = softmax_i(qt . o_i * H / 8).  Also the largest |logit|."""
    N, H = h_edge.shape[0], h_edge.shape[1] - 1
    qt_ref = torch.empty(N, 256, dtype=F64, device=DEV)
    c_ref = torch.empty(N, 256, dtype=F64, device=DEV)
    big = 0.0
    for e0, e1 in _chunks(N, H + 1):
        o = h_edge[e0:e1].double()
        qt_ref[e0:e1] = _lin(p, ATT_T, o[:, 0]) @ p[ATT_S + "weight"]
        s = torch.einsum("bd,bhd->bh", qt[e0:e1].double(), o[:, 1:]) * (H / 8.0)
        big = max(big, s.abs().max().item())
        c_ref[e0:e1] = torch.einsum("bh,bhd->bd", torch.softmax(s, dim=-1), o[:, 1:])
    return qt_ref, c_ref, big


def _node_reference(p, inp, cat):
    """From the kernel's own cat = [o_t | c]: robot_linear -> encoder_linear -> ReLU, ReLU(edge_attention_embed cat),
    the node GRU on m h_node, output_linear, the actor / critic tanh MLPs, critic_linear and fc_mean."""
    N = cat.shape[0]
    nd = "base.humanNodeRNN."
    rn = inp["robot_node"].reshape(N, 7).double()
    enc = torch.relu(_lin(p, nd + "encoder_linear.", _lin(p, "base.robot_linear.", rn)))
    emb = torch.relu(_lin(p, nd + "edge_attention_embed.", cat.double()))
    hm = inp["h_node"].reshape(N, 128).double() * inp["masks"].double().view(N, 1)
    h = _gru_step(p, nd + "gru.", torch.cat([enc, emb], 1), hm)
    y = _lin(p, nd + "output_linear.", h)
    feat = torch.tanh(_lin(p, "base.actor.2.", torch.tanh(_lin(p, "base.actor.0.", y))))
    c2 = torch.tanh(_lin(p, "base.critic.2.", torch.tanh(_lin(p, "base.critic.0.", y))))
    return {"h_node": h, "feat": feat, "value": _lin(p, "base.critic_linear.", c2), "mean": _lin(p, "dist.fc_mean.", feat)}


# ------------------------------------------------------------------------------------------------ A-C. stages vs float64
# Tolerance per mode and output, in units of max(1, max |reference|): about 2x the worst error measured on a B200 (1000 W)
# over STAGE_CASES.  h_edge is the edge stage, qt the query projection, c the attention kernel, the rest the node / heads
# stage.  Worst measured (fp32 / bf16x3 / fp16 / bf16):
#   h_edge  8.6e-6 / 5.3e-4 / 2.1e-2 / 2.7e-1    qt    7.6e-7 / 6.0e-6 / 3.5e-4 / 2.6e-3    c     7.9e-6 in any mode
#   h_node  1.9e-6 / 4.2e-5 / 2.7e-3 / 2.3e-2    feat  4.1e-6 / 5.2e-5 / 3.9e-3 / 3.3e-2
#   value   1.7e-6 / 2.3e-5 / 2.1e-3 / 1.8e-2    mean  6.6e-7 / 1.5e-5 / 8.0e-4 / 6.9e-3
# The edge stage's worst case is the x4 edge weights with zero masks (edge_x4 N=4097 H=7): its gate pre-activations are
# large sums of large terms, and every mode's error grows with them (fp32 too, 8.6e-6 there against 1e-6 elsewhere); the
# edge errors of the shipped checkpoints stay below 6e-5 in bf16x3.  Within every output but c each tolerance lies below
# the error the next weaker mode measured on the case where the stronger one measured its worst (by 3x for fp32 / bf16x3
# on qt, by 4x or more everywhere else), so a kernel that silently runs a weaker mode fails.  The attention kernel is fp32
# arithmetic in every mode (it is fed the GPU's own qt and h_edge), so c cannot separate the modes; qt, the product in
# front of it, does.
TOL = {
    "fp32": dict(h_edge=2e-5, qt=2e-6, c=2e-5, h_node=4e-6, feat=1e-5, value=4e-6, mean=2e-6),
    "bf16x3": dict(h_edge=1.1e-3, qt=1.5e-5, c=2e-5, h_node=1e-4, feat=1.1e-4, value=5e-5, mean=3e-5),
    "fp16": dict(h_edge=4.5e-2, qt=8e-4, c=2e-5, h_node=6e-3, feat=8e-3, value=4.5e-3, mean=1.6e-3),
    "bf16": dict(h_edge=0.55, qt=6e-3, c=2e-5, h_node=5e-2, feat=7e-2, value=4e-2, mean=1.4e-2),
}

STAGE_CASES = [
    # (weights, N, H, masks, inputs)
    ("holonomic_27776", 1, 1, "mixed", "synthetic"),
    ("holonomic_27776", 3, 5, "ones", "synthetic"),
    ("unicycle_55554", 129, 20, "mixed", "synthetic"),
    ("edge_x4", 129, 20, "fractional", "synthetic"),
    ("edge_x4", 65, 32, "mixed", "synthetic"),
    ("edge_x4", 4097, 7, "zeros", "synthetic"),
    ("unicycle_55554", 20000, 1, "mixed", "synthetic"),
    ("logits300", 129, 20, "ones", "synthetic"),
    ("logits300", 1024, 10, "mixed", "synthetic"),
    ("holonomic_27776", 1024, 10, "fractional", "synthetic"),
    ("edge_x4", 16384, 20, "mixed", "synthetic"),
    ("holonomic_27776", 16384, 20, "mixed", "realistic"),
    ("unicycle_55554", 65536, 20, "mixed", "synthetic"),
]


@pytest.mark.parametrize("weights,N,H,masks,inputs", STAGE_CASES)
def test_forward_stages_match_float64(policies, request, weights, N, H, masks, inputs):
    """Every mode on the same inputs through Policy.cuda_forward with a caller-owned, NaN-filled workspace:
      h_edge_out against one float64 step of both edge GRUs on the same fp32 inputs;
      qt (workspace) against W_s^T (W_t o_t + b_t) of the GPU's h_edge_out, c = cat[:, 256:] against the softmax-weighted
        sum with the GPU's qt; cat[:, :256] is a copy of h_edge_out[:, 0], bit for bit;
      h_node_out, actor_features, value and action_mean against the float64 node / heads chain on the GPU's cat."""
    policy = policies[weights]
    inp = request.getfixturevalue("realistic") if inputs == "realistic" else _synthetic(N, H, masks, seed=N * 33 + H)
    assert inp["spatial_edges"].shape[:2] == (N, H)
    p = _params64(policy)
    want_edge = _edge_reference(p, inp)
    case = "%s N=%d H=%d %s %s" % (weights, N, H, masks, inputs)
    for mode in MODES:
        got, ws = _cuda_forward(policy, inp, mode)
        tol = TOL[mode]
        what = "stage %s %s " % (case, mode)
        _check(what + "h_edge", got["h_edge"], want_edge, tol["h_edge"])
        qt, cat = _ws_views(ws, N)
        assert _same_bits(cat[:, :256], got["h_edge"][:, 0]), what + "cat[:, :256] is not h_edge_out[:, 0]"
        qt_ref, c_ref, big = _attention_reference(p, got["h_edge"], qt)
        _check(what + "qt", qt, qt_ref, tol["qt"])
        _check(what + "c", cat[:, 256:], c_ref, tol["c"])
        if weights == "logits300" and H >= 10:
            assert big >= 100.0, (what, "largest |logit|", big)
        want = _node_reference(p, inp, cat)
        for k in ("h_node", "feat", "value", "mean"):
            _check(what + k, got[k].reshape(want[k].shape), want[k], tol[k])


def test_mode_tolerances_are_ordered():
    """Each output's tolerance grows from fp32 to bf16x3 to fp16 to bf16 (c excepted: one fp32 kernel in every mode)."""
    for k in TOL["fp32"]:
        if k != "c":
            assert [TOL[m][k] for m in MODES] == sorted(TOL[m][k] for m in MODES) and len({TOL[m][k] for m in MODES}) == 4, k


# ------------------------------------------------------------------------------------------------ D. write and read discipline
GUARD_ROWS = 128      # one tile: a store that ignores the row bound of the last partial tile lands at most 127 rows late


def _guarded(rows, cols, dtype=torch.float32):
    """A [rows, cols] tensor in the middle of a buffer with GUARD_ROWS rows of NaN on either side."""
    if dtype is torch.float32:
        buf = torch.full(((rows + 2 * GUARD_ROWS) * cols,), float("nan"), device=DEV)
    else:
        buf = torch.full(((rows + 2 * GUARD_ROWS) * cols,), -1, dtype=torch.int16, device=DEV).view(dtype)
    return buf, buf[GUARD_ROWS * cols:(GUARD_ROWS + rows) * cols].view(rows, cols)


def _outside(buf, rows, cols):
    return torch.cat([buf[:GUARD_ROWS * cols], buf[(GUARD_ROWS + rows) * cols:]])


@pytest.mark.parametrize("N,H", [(1, 1), (3, 5), (129, 20), (4097, 7)])
@pytest.mark.parametrize("mode", MODES)
def test_forward_writes_only_its_outputs(policies, mode, N, H):
    """h_edge_out, h_node_out, value, mean, actor_features and the edge image are slices of NaN-filled buffers and the
    workspace is NaN-filled: every output element is written (no NaN) and nothing outside the slices changes.  Only bf16x3
    writes the image; the other modes leave it untouched.  A second forward with actor_features = NULL gives the same
    value / mean bits and writes nothing else."""
    policy = policies["edge_x4"]
    inp = _synthetic(N, H, "mixed", seed=91 + N)
    shapes = {"h_node": (N, 128), "h_edge": (N * (H + 1), 256), "value": (N, 1), "mean": (N, 2), "feat": (N, 256)}
    bufs, out = {}, {}
    for k, (r, c) in shapes.items():
        bufs[k], out[k] = _guarded(r, c)
    img = [_guarded(N * (H + 1), 256, BF16) for _ in range(2)]
    before = {k: b.clone() for k, b in bufs.items()}
    img_before = [b.clone() for b, _ in img]
    policy._ensure_handle(DEV)
    policy.set_edge_image(None, (img[0][1], img[1][1]))
    try:
        _abi_forward(policy, inp, mode, out, _workspace(N, H))
        torch.cuda.synchronize()
    finally:
        policy.set_edge_image(None, None)
    for k, (r, c) in shapes.items():
        assert not bool(out[k].isnan().any()), (mode, k, "has unwritten (or NaN-read) elements")
        assert _same_bits(_outside(bufs[k], r, c), _outside(before[k], r, c)), (mode, k, "written outside the output")
    for (buf, view), old in zip(img, img_before):
        if mode == "bf16x3":
            assert not bool(view.isnan().any()), "edge image not fully written"
            rows = N * (H + 1)
            assert _same_bits(_outside(buf, rows, 256), _outside(old, rows, 256)), "edge image written outside its rows"
        else:
            assert _same_bits(buf, old), (mode, "only bf16x3 writes the edge image")
    nofeat = {k: _guarded(*shapes[k])[1] for k in ("h_node", "h_edge", "value", "mean")}
    nofeat["feat"] = None
    _abi_forward(policy, inp, mode, nofeat, _workspace(N, H))
    torch.cuda.synchronize()
    for k in ("h_node", "h_edge", "value", "mean"):
        assert _same_bits(nofeat[k], out[k]), (mode, k, "differs with actor_features = NULL")


def test_forward_is_bitwise_repeatable_at_the_c3_shape(policies):
    """The same forward twice gives the same bits of every output in every mode at 16384 envs x 20 humans (the forward
    kernels use no atomics; GraphedRollout's replay-equals-eager tests rely on it)."""
    policy = policies["holonomic_27776"]
    N, H = 16384, 20
    inp = _synthetic(N, H, "mixed", seed=5)
    for mode in MODES:
        a, _ = _cuda_forward(policy, inp, mode)
        b, _ = _cuda_forward(policy, inp, mode)
        for k in a:
            assert _same_bits(a[k], b[k]), (mode, k)


# ------------------------------------------------------------------------------------------------ E. resident edge image
def _logical_rows(h_edge):
    """[N, H + 1, 256] -> the image's row order: spatial rows env * H + human first, then the N temporal rows."""
    N, H1 = h_edge.shape[:2]
    return torch.cat([h_edge[:, 1:].reshape(N * (H1 - 1), 256), h_edge[:, 0]], 0)


def _image_pair(rows):
    return tuple(torch.full((rows, 256), -1, dtype=torch.int16, device=DEV).view(BF16) for _ in range(2))


@pytest.mark.parametrize("N,H", [(129, 20), (16384, 20)])
def test_resident_edge_image(policies, N, H):
    """bf16x3: the image a forward writes is bf16(x), bf16(x - bf16(x)) of its h_edge_out in logical row order, bit for bit.
    The next forward (0 / 1 masks) gives the same bits of h_edge_out, h_node_out, value, mean and of its own image whether
    it reads its A operand from that image or converts the fp32 h_edge_in.  In fp32, fp16 and bf16 mode a forward neither
    writes an image that is set nor reads one: with a garbage input image it gives the bits of a forward without one."""
    policy = policies["holonomic_27776"]
    policy._ensure_handle(DEV)
    rows = N * (H + 1)
    inp1 = _synthetic(N, H, "mixed", seed=17)
    img1 = _image_pair(rows)
    try:
        policy.set_edge_image(None, img1)
        out1, _ = _cuda_forward(policy, inp1, "bf16x3")
        hi, lo = _split(_logical_rows(out1["h_edge"]))
        assert _same_bits(img1[0], hi) and _same_bits(img1[1], lo), "image is not the split of h_edge_out in logical order"
        inp2 = _synthetic(N, H, "mixed", seed=18)
        inp2["h_node"], inp2["h_edge"] = out1["h_node"], out1["h_edge"]
        assert 0 < int((inp2["masks"] == 0).sum()) < N or N < 10
        res = {}
        for way, image_in in (("image", img1), ("fp32", None)):
            img2 = _image_pair(rows)
            policy.set_edge_image(image_in, img2)
            res[way] = _cuda_forward(policy, inp2, "bf16x3")[0], img2
        (a, ia), (b, ib) = res["image"], res["fp32"]
        for k in ("h_edge", "h_node", "value", "mean", "feat"):
            assert _same_bits(a[k], b[k]), ("reading the image changes", k)
        assert _same_bits(ia[0], ib[0]) and _same_bits(ia[1], ib[1]), "reading the image changes the output image"
        garbage = tuple(torch.randn(rows, 256, device=DEV, generator=_gen(3 + i)).bfloat16() for i in range(2))
        for mode in ("fp32", "fp16", "bf16"):
            policy.set_edge_image(None, None)
            want, _ = _cuda_forward(policy, inp2, mode)
            img = _image_pair(rows)
            policy.set_edge_image(garbage, img)
            got, _ = _cuda_forward(policy, inp2, mode)
            assert bool((_bits(img[0]) == -1).all()) and bool((_bits(img[1]) == -1).all()), (mode, "wrote the edge image")
            for k in want:
                assert _same_bits(got[k], want[k]), (mode, k, "read the edge image")
    finally:
        policy.set_edge_image(None, None)


# ------------------------------------------------------------------------------------------------ F. weight re-packing
def _forward_all_modes(policy, inp):
    return {mode: _cuda_forward(policy, inp, mode)[0] for mode in MODES}


@pytest.mark.parametrize("N,H", [(129, 20), (16384, 20)])
@pytest.mark.parametrize("how", ["load_state_dict", "new_storage", "invalidate_weights"])
def test_repacked_weights_match_a_fresh_policy(how, N, H):
    """A policy that ran with weights A and then got weights B gives, in every mode, the bits of a fresh Policy built from
    B -- through every image cn_dsrnn_update_weights re-packs (edge weights, node / heads weights and constants, the linear
    layers, the folded attention product).  B arrives by load_state_dict (same storage, version bumped), as new tensors at
    new addresses, or by an edit through .data (no version bump) followed by invalidate_weights()."""
    sd_a, sd_b = dsrnn_oracle.random_state_dict(seed=41), dsrnn_oracle.random_state_dict(seed=42)
    policy = _make_policy(sd_a)
    inp = _synthetic(N, H, "mixed", seed=43)
    _forward_all_modes(policy, inp)                       # the handle exists and has run every mode with A
    params = dict(policy.named_parameters())
    if how == "load_state_dict":
        policy.load_state_dict(sd_b)
    elif how == "new_storage":
        with torch.no_grad():
            for k, t in params.items():
                t.data = sd_b[k].to(DEV).clone()
    else:
        versions = [t._version for t in params.values()]
        for k, t in params.items():
            t.data.copy_(sd_b[k])
        assert [t._version for t in params.values()] == versions          # only invalidate_weights() can tell the handle
        policy.invalidate_weights()
    got = _forward_all_modes(policy, inp)
    want = _forward_all_modes(_make_policy(sd_b), inp)
    for mode in MODES:
        for k in want[mode]:
            assert _same_bits(got[mode][k], want[mode][k]), (how, mode, k)
