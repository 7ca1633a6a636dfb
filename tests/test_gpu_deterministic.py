"""GPU: bit-reproducible native PPO update (training.cuda_deterministic) -- cn_gemm_bf16x3_ordered (split-K partial products
summed in slice order), cn_encoder_grad_ordered, and the native update / train() built on them."""
import ctypes as C
import math

import pytest
import torch

from crowdnav_dsrnn_b200 import Config, _lib, native
from crowdnav_dsrnn_b200.ppo import PPO

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def _check(got, want, tol):
    err = (got.double() - want).abs().max().item()
    assert err <= tol * max(1.0, want.abs().max().item()), (err, want.abs().max().item())


@pytest.fixture
def ordered(monkeypatch):
    monkeypatch.setattr(native, "DETERMINISTIC", True)
    assert native.ordered()


def _wgrad(rows, m, n, split, seed=7, c=None):
    """dW = dY^T X; on a given C the product is added (split problems always add; one slice needs accumulate)."""
    dy, x = _rand(rows, m, seed=seed), _rand(rows, n, seed=seed + 1)
    acc = c is not None
    c = torch.zeros(m, n, device=DEV) if c is None else c
    return dy, x, dict(a=native.split(dy), a_mn=True, b=native.split(x), b_mn=True, c=c, split_k=split, accumulate=acc)


WGRAD = [(5000, 768, 256, 0), (5000, 768, 64, 0), (130, 384, 128, 1), (70000, 256, 512, 0), (999, 100 * 8, 72, 3)]


@pytest.mark.parametrize("rows,m,n,split", WGRAD)
def test_ordered_gemm_accuracy_and_accumulate(ordered, rows, m, n, split):
    """dW = dY^T X with ordered split-K: within 3e-5 of float64; on an initialised C it adds the product (C0 + A B)."""
    dy, x, p = _wgrad(rows, m, n, split)
    native.gemm([p])
    want = dy.double().t() @ x.double()
    _check(p["c"], want, 3e-5)
    c0 = _rand(m, n, seed=9)
    _, _, p = _wgrad(rows, m, n, split, c=c0.clone())
    native.gemm([p])
    _check(p["c"], c0.double() + want, 3e-5)


def test_ordered_gemm_grouped_launch(ordered):
    """Four problems of different shape / major in one ordered launch (two of them split)."""
    xs = [_rand(500, 128, seed=10), _rand(64, 768, seed=11), _rand(3000, 384, seed=12), _rand(20000, 72, seed=13)]
    ws = [_rand(256, 128, seed=14), _rand(768, 256, seed=15), _rand(3000, 128, seed=16), _rand(20000, 1024, seed=17)]
    cs = [torch.empty(500, 256, device=DEV), torch.empty(64, 256, device=DEV), torch.zeros(384, 128, device=DEV),
          torch.full((72, 1024), 0.5, device=DEV)]
    native.gemm([dict(a=native.split(xs[0]), b=native.split(ws[0]), c=cs[0]),
                 dict(a=native.split(xs[1]), b=native.split(ws[1]), b_mn=True, c=cs[1]),
                 dict(a=native.split(xs[2]), a_mn=True, b=native.split(ws[2]), b_mn=True, c=cs[2], split_k=0),
                 dict(a=native.split(xs[3]), a_mn=True, b=native.split(ws[3]), b_mn=True, c=cs[3], split_k=0)])
    _check(cs[0], xs[0].double() @ ws[0].double().t(), 2e-5)
    _check(cs[1], xs[1].double() @ ws[1].double(), 2e-5)
    _check(cs[2], xs[2].double().t() @ ws[2].double(), 3e-5)
    _check(cs[3], 0.5 + xs[3].double().t() @ ws[3].double(), 3e-5)


@pytest.mark.parametrize("rows,m,n,split", WGRAD)
def test_ordered_gemm_is_bitwise_stable(ordered, rows, m, n, split):
    """Five launches give the same bits; so does the problem launched alone and grouped with three others."""
    _, _, p = _wgrad(rows, m, n, split)
    native.gemm([p])
    first = p["c"].clone()
    for _ in range(4):
        p["c"].zero_()
        native.gemm([p])
        assert torch.equal(p["c"], first)
    others = [_wgrad(4000, 256, 128, 0, seed=40)[2], _wgrad(777, 64, 72, 2, seed=42)[2], _wgrad(30000, 1024, 72, 0, seed=44)[2]]
    p["c"].zero_()
    native.gemm([others[0], p, others[1], others[2]])
    assert torch.equal(p["c"], first)
    assert native.ordered_workspace([p])[1][0] == native.ordered_workspace([others[0], p, others[1], others[2]])[1][1]


@pytest.mark.parametrize("rows,m,n,split", WGRAD)
def test_ordered_gemm_agrees_with_atomic_split_k(rows, m, n, split):
    """The ordered mode computes the same product as the default (atomic) mode, only summed in a fixed order."""
    _, _, p = _wgrad(rows, m, n, split)
    native.gemm([p])
    atomic = p["c"].clone()
    p["c"].zero_()
    native.DETERMINISTIC = True
    try:
        native.gemm([p])
    finally:
        native.DETERMINISTIC = False
    assert (p["c"] - atomic).abs().max().item() <= 1e-5 * atomic.abs().max().item()


def test_ordered_entry_points_refuse_bad_workspaces():
    """A NULL, too small or misaligned workspace is refused and nothing is launched (C keeps its value)."""
    lib = _lib.load()
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    _, _, p = _wgrad(5000, 768, 64, 0)
    p["c"].fill_(7.0)
    need, slices = native.ordered_workspace([p])
    assert slices[0] > 1 and need == slices[0] * 768 * 64 * 4
    arr, _, _ = native._gemm_array([p])
    ws = torch.empty(need + 64, dtype=torch.uint8, device=DEV)
    for ptr, size in ((None, need), (ws.data_ptr(), need - 4), (ws.data_ptr() + 16, need)):
        assert lib.cn_gemm_bf16x3_ordered(arr, 1, C.c_void_p(ptr) if ptr else None, size, stream) != 0
        assert b"workspace" in lib.cn_last_error()
    de, x = _rand(1000, 64, seed=50), _rand(1000, 2, seed=51)
    e_hi = _rand(1000, 64, seed=52).bfloat16()
    dw, db = torch.full((64, 2), 7.0, device=DEV), torch.full((64,), 7.0, device=DEV)
    nbytes = lib.cn_encoder_grad_ordered_workspace_bytes(1000)
    assert nbytes == 250 * 192 * 4
    for ptr, size in ((None, nbytes), (ws.data_ptr(), nbytes - 4)):
        assert lib.cn_encoder_grad_ordered(C.c_void_p(de.data_ptr()), C.c_void_p(e_hi.data_ptr()), 64, C.c_void_p(x.data_ptr()),
                                           C.c_void_p(dw.data_ptr()), C.c_void_p(db.data_ptr()), 1000,
                                           C.c_void_p(ptr) if ptr else None, size, stream) != 0
    torch.cuda.synchronize()
    assert bool((p["c"] == 7.0).all()) and bool((dw == 7.0).all()) and bool((db == 7.0).all())


@pytest.mark.parametrize("rows", [3, 1000, 123457])
def test_ordered_encoder_grad_matches_float64_and_is_bitwise_stable(ordered, rows):
    de, x = _rand(rows, 64, seed=60), _rand(rows, 2, seed=61)
    e = _rand(rows, 72, seed=62)
    e_hi = e.bfloat16()
    on = (e_hi[:, :64].float() > 0).double()
    want_w = (de.double() * on).t() @ x.double()
    want_b = (de.double() * on).sum(0)
    dw0, db0 = _rand(64, 2, seed=63), _rand(64, seed=64)
    first = None
    for _ in range(5):
        dw, db = dw0.clone(), db0.clone()
        native.encoder_grad(de, e_hi, 72, x, dw, db)
        if first is None:
            first = (dw, db)
            _check(dw, dw0.double() + want_w, 2e-5)
            _check(db, db0.double() + want_b, 2e-5)
        else:
            assert torch.equal(dw, first[0]) and torch.equal(db, first[1])


def _pass_grads(policy, obs, h0, masks, action):
    policy.zero_grad(set_to_none=True)
    value, logp, ent, _ = policy.evaluate_actions(obs, {k: v.clone() for k, v in h0.items()}, masks, action)
    (value.mean() + logp.mean() - 0.01 * ent).backward()
    return {k: q.grad.clone() for k, q in policy.named_parameters() if q.grad is not None}


def test_native_gradients_are_bitwise_reproducible_in_ordered_mode(ordered):
    """Race detector at zero tolerance: eight native forward + backward passes give identical gradients."""
    from test_config_host import _sequence_case

    policy, obs, masks, action, h0 = _sequence_case(torch.float32, DEV, n=40, H=20, T=5, seed=3)
    policy.sequence_impl = "native"
    first = _pass_grads(policy, obs, h0, masks, action)
    assert len(first) >= 40
    for rep in range(1, 8):
        grads = _pass_grads(policy, obs, h0, masks, action)
        bad = [k for k in first if not torch.equal(grads[k], first[k])]
        assert not bad, (rep, bad)


def test_ordered_mode_follows_torch_deterministic_algorithms():
    assert not native.ordered()
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        assert native.ordered()
    finally:
        torch.use_deterministic_algorithms(prev)


def test_ppo_update_native_deterministic_matches_reference_golden():
    """PPO(native=True, deterministic=True) against the reference's own PPO.update within the same 2 %; the flag is scoped
    to the update."""
    from test_ppo_update import _check_update, _golden, _policy, _storage

    g = _golden()
    hyper = g["hyper"]
    policy = _policy().to(DEV)
    before = {k: v.detach().cpu().clone() for k, v in policy.state_dict().items()}
    st = _storage(g, keep_hidden_history=False).to(DEV)
    st.compute_returns(torch.from_numpy(g["next_value"]).to(DEV), True, float(hyper[8]), float(hyper[9]), False)
    agent = PPO(policy, float(hyper[0]), int(hyper[1]), int(hyper[2]), float(hyper[3]), float(hyper[4]), lr=float(hyper[5]),
                eps=float(hyper[6]), max_grad_norm=float(hyper[7]), native=True, deterministic=True)
    torch.manual_seed(int(hyper[10]))
    launches = native.COUNTERS["gemm_launches"]
    losses = agent.update(st)
    assert native.COUNTERS["gemm_launches"] > launches + 100 and not native.DETERMINISTIC
    cpu_policy = _policy()
    cpu_policy.load_state_dict({k: v.detach().cpu() for k, v in policy.state_dict().items()})
    _check_update(g, cpu_policy, before, losses)


def test_native_pass_at_the_benchmark_shape():
    """One native forward + backward at 4096 envs x 20 humans x T = 30 (the c5 update's pass) on seeded synthetic rollout
    data: ordered mode twice gives identical gradients, and agrees with the default mode within 1e-3 of each scale (the
    accuracy the native gradients are held to against the fp32 torch graph).  Not tighter: in the default mode the temporal
    GRU's weight gradients (122880 rows, grouped with the 20x larger spatial ones) get one k-slice, in ordered mode 48, and
    the two summation orders differ by up to 4.6e-4 of those gradients' scale on this data (B200); the gradients of every
    other parameter agree to 2.5e-5."""
    from crowdnav_dsrnn_b200.model import Policy
    from crowdnav_dsrnn_b200.spaces import crowd_spaces

    n, H, T = 4096, 20, 30
    obs_space, act_space = crowd_spaces(H)
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        policy = Policy(obs_space.spaces, act_space, base="srnn", base_kwargs=Config(human_num=H)).to(DEV)
    policy.sequence_impl = "native"
    g = torch.Generator(device=DEV).manual_seed(0)
    obs = {"robot_node": torch.randn(T * n, 1, 7, device=DEV, generator=g),
           "temporal_edges": torch.randn(T * n, 1, 2, device=DEV, generator=g),
           "spatial_edges": torch.randn(T * n, H, 2, device=DEV, generator=g) * 3}
    masks = (torch.rand(T * n, 1, device=DEV, generator=g) > 0.03).float()
    action = torch.randn(T * n, 2, device=DEV, generator=g)
    h0 = {"human_node_rnn": torch.randn(n, 1, 128, device=DEV, generator=g) * 0.3,
          "human_human_edge_rnn": torch.randn(n, H + 1, 256, device=DEV, generator=g) * 0.3}
    default = _pass_grads(policy, obs, h0, masks, action)
    native.DETERMINISTIC = True
    try:
        a = _pass_grads(policy, obs, h0, masks, action)
        b = _pass_grads(policy, obs, h0, masks, action)
    finally:
        native.DETERMINISTIC = False
    assert sorted(a) == sorted(default) and len(a) >= 40
    assert not [k for k in a if not torch.equal(a[k], b[k])]
    bad = [k for k in a if (a[k] - default[k]).abs().max().item() > 1e-3 * max(default[k].abs().max().item(), 1e-3)]
    assert not bad, bad


def test_train_with_cuda_deterministic_is_reproducible(tmp_path):
    """train() twice with training.cuda_deterministic and the native update: the last checkpoints hold identical tensors
    and the history rows agree in everything but fps."""
    from crowdnav_dsrnn_b200.train import train

    runs = []
    for tag in ("a", "b"):
        cfg = Config(human_num=5)
        cfg.training.num_processes = 256
        cfg.ppo.num_steps = 8
        cfg.training.cuda_deterministic = True
        _, history = train(cfg, DEV, num_updates=3, output_dir=str(tmp_path / tag), log=None, native_update=True)
        runs.append((torch.load(tmp_path / tag / "checkpoints" / "00002.pt", map_location="cpu"), history))
    (sd_a, hist_a), (sd_b, hist_b) = runs
    assert sorted(sd_a) == sorted(sd_b)
    assert not [k for k in sd_a if not torch.equal(sd_a[k], sd_b[k])]
    strip = lambda rows: [{k: v for k, v in r.items() if k != "fps"} for r in rows]
    same = lambda x, y: x == y or (isinstance(x, float) and isinstance(y, float) and math.isnan(x) and math.isnan(y))
    assert len(hist_a) == 3 and all(same(r[k], s[k]) for r, s in zip(strip(hist_a), strip(hist_b)) for k in r)
