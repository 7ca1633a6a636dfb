"""GPU: the kernels of the native PPO update one by one against float64 references -- the training instantiation of the
tcgen05 edge-GRU kernel (cn_dsrnn_edge_sequence_step), cn_gru_gates_backward_pairs, cn_encoder_grad (atomic),
cn_attention_train_forward / _backward and cn_gemm_bf16x3 at the products of the c5 update -- and the whole native pass at
the benchmark shape against the same policy evaluated in float64.

Every reference is plain torch in float64 on the GPU.  Each check prints its worst error next to its tolerance (run with -s
to see the margins)."""
import copy
import ctypes as C

import pytest
import torch

from crowdnav_dsrnn_b200 import Config, _lib, abi, native

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
F64 = torch.float64
BF16 = torch.bfloat16


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _randn(*shape, seed, scale=1.0):
    return torch.randn(*shape, device=DEV, generator=_gen(seed)) * scale


def _check(name, got, want, tol, floor=1.0):
    """max |got - want| <= tol * max(floor, max |want|); a NaN in `got` fails."""
    scale = max(floor, want.abs().max().item())
    err = (got.double() - want).abs().max().item()
    print("%-48s err %.3e of scale %.3e = %.2e (tol %.1e)" % (name, err, scale, err / scale, tol))
    assert err <= tol * scale, (name, err, scale)


def _check_elementwise(name, got, want, bound):
    """|got - want| <= bound element by element; reports the worst ratio."""
    ratio = ((got.double() - want).abs() / bound).max().item()
    print("%-48s worst error / bound %.3f" % (name, ratio))
    assert ratio <= 1.0, (name, ratio)


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _split_is_canonical(hi, lo):
    """hi is a nearest bfloat16 of hi + lo, i.e. (hi, lo) is what bf16(x), bf16(x - bf16(x)) gives for some fp32 x.
    hi == bf16(hi + lo) except where hi + lo is an exact tie between two bf16 values; then |lo| is half the spacing."""
    s = hi.float() + lo.float()                       # exact: hi and lo have 8-bit mantissas at least 8 bits apart
    back = s.bfloat16()
    same = _bits(back) == _bits(hi)
    tie = (back.float() - hi.float()).abs() == 2 * lo.float().abs()
    return bool((same | tie).all())


# ------------------------------------------------------------------------------------------------ A. edge GRU sequence step
@pytest.fixture(scope="module")
def edge_policy():
    """A seeded Policy whose edge-GRU weights are scaled up (x4) so that the gates spread over their whole range instead
    of sitting near 0.5; the edge weights do not depend on human_num, so one handle serves every H."""
    from crowdnav_dsrnn_b200.model import Policy
    from crowdnav_dsrnn_b200.spaces import crowd_spaces

    obs_space, act_space = crowd_spaces(5)
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(2024)
        policy = Policy(obs_space.spaces, act_space, base="srnn", base_kwargs=Config(human_num=5)).to(DEV)
    b = policy.base
    with torch.no_grad():
        for mod in (b.humanhumanEdgeRNN_spatial.gru, b.humanhumanEdgeRNN_temporal.gru):
            for p in mod.parameters():
                p.mul_(4.0)
    policy._ensure_handle(DEV)
    return policy


def _edge_params(policy, spatial):
    m = policy.base.humanhumanEdgeRNN_spatial if spatial else policy.base.humanhumanEdgeRNN_temporal
    return {k: v.detach().double() for k, v in (("enc_w", m.encoder_linear.weight), ("enc_b", m.encoder_linear.bias),
                                                ("w_ih", m.gru.weight_ih_l0), ("w_hh", m.gru.weight_hh_l0),
                                                ("b_ih", m.gru.bias_ih_l0), ("b_hh", m.gru.bias_hh_l0))}


def _edge_reference(p, x, h_in, m_rows):
    """One step of one edge GRU in float64: e = ReLU(W_enc x + b), hm = m h_in, the torch.nn.GRU step (gate order r|z|n),
    h = n + z (hm - n).  Also returns |W_enc| |x| + |b|, the magnitude the fp32 encoder rounds against."""
    x64 = x.double()
    e = torch.relu(x64 @ p["enc_w"].t() + p["enc_b"])
    cond = x64.abs() @ p["enc_w"].abs().t() + p["enc_b"].abs()
    hm = (h_in * m_rows[:, None]).double()                 # m is 0 / 1: the fp32 product is exact
    gi = e @ p["w_ih"].t() + p["b_ih"]
    gh = hm @ p["w_hh"].t() + p["b_hh"]
    r = torch.sigmoid(gi[:, :256] + gh[:, :256])
    z = torch.sigmoid(gi[:, 256:512] + gh[:, 256:512])
    hn = gh[:, 512:]
    n = torch.tanh(gi[:, 512:] + r * hn)
    return dict(e=e, cond=cond, r=r, z=z, n=n, hn=hn, h=n + z * (hm - n))


def _edge_masks(kind, n, seed):
    if kind == "zeros":
        return torch.zeros(n, device=DEV)
    if kind == "ones":
        return torch.ones(n, device=DEV)
    return (torch.rand(n, device=DEV, generator=_gen(seed)) > 0.2).float()


EDGE_CASES = [(1, 1, "mixed"), (3, 1, "mixed"), (7, 32, "mixed"), (129, 20, "mixed"), (1000, 5, "mixed"), (20000, 1, "mixed"),
              (4096, 20, "mixed"), (7, 32, "zeros"), (129, 20, "ones"), (4096, 20, "zeros"), (4096, 20, "ones")]


@pytest.mark.parametrize("n,H,masks", EDGE_CASES)
def test_edge_sequence_step_outputs_match_float64(edge_policy, n, H, masks):
    """Steps t = 1 and t = 2 of a T = 3 sequence layout ([T*S spatial | T*n temporal] rows): step 1 reads the t = 0 rows,
    step 2 the rows step 1 wrote.  Every other row of every buffer starts as NaN (fp32) / 0xFFFF (bf16): a read of a row
    the step must not read turns its outputs into NaN, and a write outside [out_row, +rows) of either problem changes
    bits that must stay.  Checked against float64:
      h_out and r | z | n | W_hn hm + b_hn in ws: 1.5e-4 of the scale.  The bf16x3 products carry 2^-16 relative operand
        error over K = 320 and the gates use ex2 / rcp approximations; with the x4 weights of `edge_policy` the worst errors
        measured on a B200 were 8.4e-5 (n in ws) and 5.9e-5 (h_out), both at n = 4096, H = 20, above the 5e-5 the forward
        GEMM tests use;
      hm_hi / hm_lo: bit-equal to bf16(x) and bf16(x - hi) of the fp32 masked state x = m h_in;
      e_hi + e_lo: within 2^-16 |e| plus 2^-22 (|W_enc| |x| + |b|) (the fp32 rounding of the encoder) of the float64 e;
      e_hi exactly zero wherever e is below zero by more than that rounding (cn_encoder_grad reads the ReLU sign from it);
      columns 64..71 of e_hi are [1, 0 x 7] and of e_lo zero."""
    lib = _lib.load()
    T, S = 3, n * H
    rows = T * (S + n)
    hs = torch.full((rows, 256), float("nan"), device=DEV)
    hs[:S] = _randn(S, 256, seed=1, scale=0.7)                        # the rows step 0 would have written
    hs[T * S:T * S + n] = _randn(n, 256, seed=2, scale=0.7)
    ws = torch.full((rows, 1024), float("nan"), device=DEV)
    hm_hi, hm_lo = (torch.full((rows, 256), -1, dtype=torch.int16, device=DEV).view(BF16) for _ in range(2))
    e_hi, e_lo = (torch.full((rows, 72), -1, dtype=torch.int16, device=DEV).view(BF16) for _ in range(2))
    bufs = (hs, ws, hm_hi, hm_lo, e_hi, e_lo)
    p_s, p_t = _edge_params(edge_policy, True), _edge_params(edge_policy, False)
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    for t in (1, 2):
        te = _randn(n, 2, seed=10 * t)
        se = _randn(S, 2, seed=10 * t + 1, scale=3.0)
        mk = _edge_masks(masks, n, seed=10 * t + 2)
        in_s, in_t = (t - 1) * S, T * S + (t - 1) * n
        out_s, out_t = t * S, T * S + t * n
        before = [b.clone() for b in bufs]
        io = abi.CnEdgeSeqStep()
        io.temporal_edges, io.spatial_edges, io.masks, io.h_in = native._ptr(te), native._ptr(se), native._ptr(mk), native._ptr(hs)
        io.in_row_spatial, io.in_row_temporal, io.out_row_spatial, io.out_row_temporal = in_s, in_t, out_s, out_t
        io.h_out, io.ws = native._ptr(hs), native._ptr(ws)
        io.hm_hi, io.hm_lo, io.e_hi, io.e_lo = native._ptr(hm_hi), native._ptr(hm_lo), native._ptr(e_hi), native._ptr(e_lo)
        _lib.check(lib.cn_dsrnn_edge_sequence_step(edge_policy._handle, n, H, C.byref(io), stream), "cn_dsrnn_edge_sequence_step")
        torch.cuda.synchronize()
        for name, old, new in zip(("h_out", "ws", "hm_hi", "hm_lo", "e_hi", "e_lo"), before, bufs):
            old[out_s:out_s + S] = new[out_s:out_s + S]
            old[out_t:out_t + n] = new[out_t:out_t + n]
            assert torch.equal(_bits(old), _bits(new)), "step %d wrote %s outside its rows" % (t, name)
        for tag, p, x, r_in, r_out, R, m_rows in (("spatial", p_s, se, in_s, out_s, S, mk.repeat_interleave(H)),
                                                  ("temporal", p_t, te, in_t, out_t, n, mk)):
            h_in = before[0][r_in:r_in + R]
            ref = _edge_reference(p, x, h_in, m_rows)
            out = slice(r_out, r_out + R)
            what = "edge step %d %s n=%d H=%d %s" % (t, tag, n, H, masks)
            _check(what + " h_out", hs[out], ref["h"], 1.5e-4)
            for k, name in enumerate(("r", "z", "n", "hn")):
                _check(what + " ws." + name, ws[out, 256 * k:256 * (k + 1)], ref[name], 1.5e-4)
            x32 = h_in * m_rows[:, None]
            hi = x32.bfloat16()
            lo = (x32 - hi.float()).bfloat16()
            assert torch.equal(_bits(hm_hi[out]), _bits(hi)) and torch.equal(_bits(hm_lo[out]), _bits(lo)), what + " hm_hi / hm_lo"
            eh, el = e_hi[out, :64].float(), e_lo[out, :64].float()
            rnd = 2.0 ** -22 * ref["cond"]
            _check_elementwise(what + " e_hi + e_lo", eh + el, ref["e"], 2.0 ** -16 * ref["e"] + rnd)
            neg = ref["e"] == 0
            neg &= (x.double() @ p["enc_w"].t() + p["enc_b"]) < -rnd
            assert bool((eh >= 0).all()) and bool((eh[neg] == 0).all()) and bool((el[neg] == 0).all()), what + " ReLU sign of e_hi"
            tail = _bits(e_hi[out, 64:]).long()
            assert bool((tail[:, 0] == 0x3F80).all()) and bool((tail[:, 1:] == 0).all()), what + " ones column of e_hi"
            assert bool((_bits(e_lo[out, 64:]) == 0).all()), what + " ones column of e_lo"


# ------------------------------------------------------------------------------------------------ B. gate gradients
def _gates_inputs(rows, hid, seed):
    """ws = r | z | n | W_hn hm + b_hn from a float64 GRU step on random pre-activations, rounded to fp32."""
    pre = _randn(rows, 4 * hid, seed=seed, scale=2.0).double()
    r = torch.sigmoid(pre[:, :hid])
    z = torch.sigmoid(pre[:, hid:2 * hid])
    hn = pre[:, 3 * hid:]
    n = torch.tanh(pre[:, 2 * hid:3 * hid] + r * hn)
    return torch.cat([r, z, n, hn], 1).float().contiguous()


@pytest.mark.parametrize("rows", [1, 77, 4099, 86016])
@pytest.mark.parametrize("hid", [4, 12, 256])
@pytest.mark.parametrize("d_live", [0, 1])
@pytest.mark.parametrize("with_h_prev", [False, True])
def test_gru_gates_backward_pairs_matches_float64(rows, hid, d_live, with_h_prev):
    """G = [pn | pr | pz | pn r] and d = g z with g = grad_h + m_next d_in, hm = m_cur h_prev (zero state without h_prev):
    hi + lo within 2^-16 |G| plus 2^-20 of the magnitude of the terms G is formed from (fp32 rounding of the kernel's
    arithmetic, which matters where (hm - n) or (1 - n^2) cancel); hi is a nearest bf16 of hi + lo; d in place within
    2^-20 of that magnitude.  With d_live = 0 the incoming d is NaN (must not be read); one extra row after each output
    must stay untouched."""
    lib = _lib.load()
    ws = _gates_inputs(rows, hid, seed=rows + hid)
    grad_h = _randn(rows, hid, seed=1)
    d_in = _randn(rows, hid, seed=2)
    m_next = (torch.rand(rows, device=DEV, generator=_gen(3)) > 0.2).float()
    h_prev = _randn(rows, hid, seed=4, scale=0.7) if with_h_prev else None
    m_cur = (torch.rand(rows, device=DEV, generator=_gen(5)) > 0.3).float() if with_h_prev else None
    d = torch.full((rows + 1, hid), float("nan"), device=DEV)
    if d_live:
        d[:rows] = d_in
    g_hi, g_lo = (torch.full((rows + 1, 4 * hid), -1, dtype=torch.int16, device=DEV).view(BF16) for _ in range(2))
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    P = native._ptr
    _lib.check(lib.cn_gru_gates_backward_pairs(P(grad_h), P(d), d_live, P(m_next) if d_live else None, P(ws), P(h_prev), P(m_cur),
                                               P(g_hi), P(g_lo), rows, hid, stream), "cn_gru_gates_backward_pairs")
    torch.cuda.synchronize()
    assert bool(d[rows].isnan().all()) and bool((_bits(g_hi[rows]) == -1).all()) and bool((_bits(g_lo[rows]) == -1).all())
    w = ws.double()
    r, z, n, hn = w[:, :hid], w[:, hid:2 * hid], w[:, 2 * hid:3 * hid], w[:, 3 * hid:]
    g, ga = grad_h.double(), grad_h.double().abs()
    if d_live:
        g = g + m_next.double()[:, None] * d_in.double()
        ga = ga + (m_next.double()[:, None] * d_in.double()).abs()
    hp = (h_prev.double() * m_cur.double()[:, None]) if with_h_prev else torch.zeros_like(g)
    pn = g * (1 - z) * (1 - n * n)
    pn_a = ga * (1 + z) * (1 + n * n)
    G = torch.cat([pn, pn * hn * r * (1 - r), g * (hp - n) * z * (1 - z), pn * r], 1)
    Ga = torch.cat([pn_a, pn_a * hn.abs() * r * (1 + r), ga * (hp.abs() + n.abs()) * z * (1 + z), pn_a * r], 1)
    what = "gates_backward_pairs rows=%d hid=%d live=%d h_prev=%d" % (rows, hid, d_live, with_h_prev)
    hi, lo = g_hi[:rows], g_lo[:rows]
    _check_elementwise(what + " G", hi.float() + lo.float(), G, 2.0 ** -16 * G.abs() + 2.0 ** -20 * Ga + 1e-30)
    assert _split_is_canonical(hi, lo), what + " hi is not the rounding of hi + lo"
    _check_elementwise(what + " d", d[:rows], g * z, 2.0 ** -20 * ga * z + 1e-30)


# ------------------------------------------------------------------------------------------------ C. encoder gradient (atomic)
def _encoder_e_hi(rows, ld_e, seed):
    """bf16 image of e with exact zeros, negative zeros, negatives and the smallest bf16 subnormals of both signs mixed in;
    the padding columns beyond 64 hold positive values that must be ignored."""
    e = _randn(rows, ld_e, seed=seed).bfloat16()
    v = e.view(torch.int16)
    v[:, 0:64:7] = 0
    v[:, 1:64:11] = 1                       # 2^-133: the smallest positive bf16 subnormal
    v[:, 2:64:13] = -32768                  # -0
    v[:, 3:64:17] = -32767                  # -2^-133
    if ld_e > 64:
        v[:, 64:] = 0x3F80
    return e


@pytest.mark.parametrize("rows", [1, 3, 4, 5, 1000, 123457, 2457600])
@pytest.mark.parametrize("ld_e", [64, 72, 136])
def test_encoder_grad_atomic_matches_float64(rows, ld_e):
    """Default (atomic) cn_encoder_grad on non-zero dw / db: within 2e-5 of the scale of float64 (fp32 block sums added
    with atomics).  At 2 457 600 rows (the spatial rows of a c5 update) the ordered form agrees within 1e-5 of the scale."""
    assert not native.ordered()
    de, x = _randn(rows, 64, seed=60), _randn(rows, 2, seed=61)
    e_hi = _encoder_e_hi(rows, ld_e, seed=62)
    on = (e_hi[:, :64].float() > 0).double()
    assert bool((on[:, 1] == 1).all())                   # the reference counts the subnormals as positive
    dw0, db0 = _randn(64, 2, seed=63), _randn(64, seed=64)
    want_w = dw0.double() + (de.double() * on).t() @ x.double()
    want_b = db0.double() + (de.double() * on).sum(0)
    dw, db = dw0.clone(), db0.clone()
    native.encoder_grad(de, e_hi, ld_e, x, dw, db)
    _check("encoder_grad rows=%d ld_e=%d dw" % (rows, ld_e), dw, want_w, 2e-5)
    _check("encoder_grad rows=%d ld_e=%d db" % (rows, ld_e), db, want_b, 2e-5)
    if rows == 2457600:
        dwo, dbo = dw0.clone(), db0.clone()
        native.DETERMINISTIC = True
        try:
            native.encoder_grad(de, e_hi, ld_e, x, dwo, dbo)
        finally:
            native.DETERMINISTIC = False
        _check("encoder_grad ordered vs atomic dw", dwo, dw.double(), 1e-5)
        _check("encoder_grad ordered vs atomic db", dbo, db.double(), 1e-5)


# ------------------------------------------------------------------------------------------------ D. attention
def _attn_forward(o, qt, cst, scale):
    B, H = o.shape[0], o.shape[1]
    c = torch.full((B, 256), float("nan"), device=DEV)
    alpha = torch.full((B, H), float("nan"), device=DEV)
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    P = native._ptr
    _lib.check(_lib.load().cn_attention_train_forward(P(o), P(qt), P(cst), P(c), P(alpha), float(scale), B, H, stream),
               "cn_attention_train_forward")
    return c, alpha


def _attn_backward(o, qt, alpha, dc, scale, d_o, d_qt, d_cst):
    B, H = o.shape[0], o.shape[1]
    stream = C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    P = native._ptr
    _lib.check(_lib.load().cn_attention_train_backward(P(o), P(qt), P(alpha), P(dc), P(d_o), P(d_qt), P(d_cst), float(scale), B, H,
                                                       stream), "cn_attention_train_backward")


def _attn_reference(o, qt, cst, dc, scale):
    od, qd, cd = (t.double().requires_grad_(True) for t in (o, qt, cst))
    s = ((od * qd.unsqueeze(1)).sum(-1) + cd.unsqueeze(1)) * scale
    alpha = torch.softmax(s, dim=-1)
    c = (alpha.unsqueeze(-1) * od).sum(1)
    grads = torch.autograd.grad(c, (od, qd, cd), dc.double())
    a = alpha.detach()
    da = (o.double() * dc.double().unsqueeze(1)).sum(-1)                   # o_i . dc
    mag = (a * da.abs()).sum(-1) * abs(scale)                              # magnitude of the terms of sum_i alpha_i o_i . dc
    return (c.detach(), a) + grads + (s.detach(), mag)


def _attn_case(B, H, seed, logit=None):
    o = _randn(B, H, 256, seed=seed)
    qt = _randn(B, 256, seed=seed + 1, scale=0.2)
    cst = _randn(B, seed=seed + 2)
    scale = H / 8.0
    if logit is not None:                   # rescale so that the largest |logit| after scaling is exactly `logit`
        qt, cst = qt * 12.0, cst * 40.0
        s = ((o.double() * qt.double().unsqueeze(1)).sum(-1) + cst.double().unsqueeze(1)) * scale
        f = logit / s.abs().max().item()
        qt, cst = (qt * f).contiguous(), (cst * f).contiguous()
    return o, qt, cst, _randn(B, 256, seed=seed + 3), scale


def _attn_compare(what, o, qt, cst, dc, scale, tol):
    c, alpha = _attn_forward(o, qt, cst, scale)
    d_o, d_qt = torch.empty_like(o), torch.empty_like(qt)
    d_cst = torch.empty(o.shape[0], device=DEV)
    _attn_backward(o, qt, alpha, dc, scale, d_o, d_qt, d_cst)
    torch.cuda.synchronize()
    ref = _attn_reference(o, qt, cst, dc, scale)
    for name, got, want in zip(("c", "alpha", "d_o", "d_qt"), (c, alpha, d_o, d_qt), ref[:4]):
        assert bool(got.isfinite().all()), (what, name)
        _check("%s %s" % (what, name), got, want, tol)
    # d_cst = sum_i dL/ds_i = scale (sum_i alpha_i o_i.dc - sum_i alpha_i o_i.dc) is exactly zero (the softmax ignores a
    # per-sample constant): what the kernel returns is the rounding of that difference, held to `tol` of the magnitude
    # scale sum_i alpha_i |o_i.dc| of its terms
    assert bool(d_cst.isfinite().all()), (what, "d_cst")
    _check_elementwise(what + " d_cst", d_cst, ref[4], tol * ref[6] + 1e-30)
    return ref[5]


@pytest.mark.parametrize("B,H", [(122880, 20), (1001, 7), (4097, 32), (3, 1)])
def test_attention_matches_float64(B, H):
    """Forward (c, alpha) and backward (d_o, d_qt) against float64 autograd within 5e-5 of each scale, d_cst (exactly zero)
    within 5e-5 of the magnitude of the terms it cancels, at the batch of the c5 update (T n = 122880, H = 20) and at odd
    batches that leave the last block of four warps partly idle."""
    o, qt, cst, dc, scale = _attn_case(B, H, seed=B + H)
    _attn_compare("attention B=%d H=%d" % (B, H), o, qt, cst, dc, scale, 5e-5)


def test_attention_null_cst_equals_zero_cst():
    """cst = NULL is the same computation as cst = 0: identical bits of c and alpha."""
    o, qt, _, _, scale = _attn_case(1001, 7, seed=5)
    c0, a0 = _attn_forward(o, qt, torch.zeros(1001, device=DEV), scale)
    c1, a1 = _attn_forward(o, qt, None, scale)
    torch.cuda.synchronize()
    assert torch.equal(c0, c1) and torch.equal(a0, a1)


def test_attention_backward_without_d_cst_writes_only_d_o_and_d_qt():
    """With d_cst = NULL the backward writes d_o and d_qt (the same bits as with d_cst given) and nothing else: d_o and d_qt
    are carved out of one NaN-filled buffer and the gaps between and after them must stay NaN."""
    B, H = 1001, 7
    o, qt, cst, dc, scale = _attn_case(B, H, seed=6)
    c, alpha = _attn_forward(o, qt, cst, scale)
    want_o, want_q, d_cst = torch.empty_like(o), torch.empty_like(qt), torch.empty(B, device=DEV)
    _attn_backward(o, qt, alpha, dc, scale, want_o, want_q, d_cst)
    n_o, n_q, gap = B * H * 256, B * 256, 1024
    pool = torch.full((n_o + n_q + 3 * gap,), float("nan"), device=DEV)
    d_o = pool[gap:gap + n_o].view(B, H, 256)
    d_qt = pool[2 * gap + n_o:2 * gap + n_o + n_q].view(B, 256)
    _attn_backward(o, qt, alpha, dc, scale, d_o, d_qt, None)
    torch.cuda.synchronize()
    assert torch.equal(d_o, want_o) and torch.equal(d_qt, want_q)
    rest = torch.cat([pool[:gap], pool[gap + n_o:2 * gap + n_o], pool[2 * gap + n_o + n_q:]])
    assert bool(rest.isnan().all())


def test_attention_single_human_is_the_identity():
    """H = 1: alpha = 1 and c = o exactly, d_o = dc and d_qt = d_cst = 0 exactly."""
    B = 1001
    o, qt, cst, dc, scale = _attn_case(B, 1, seed=7)
    c, alpha = _attn_forward(o, qt, cst, scale)
    d_o, d_qt, d_cst = torch.empty_like(o), torch.empty_like(qt), torch.empty(B, device=DEV)
    _attn_backward(o, qt, alpha, dc, scale, d_o, d_qt, d_cst)
    torch.cuda.synchronize()
    assert bool((alpha == 1).all()) and torch.equal(c, o[:, 0])
    assert torch.equal(d_o[:, 0], dc) and bool((d_qt == 0).all()) and bool((d_cst == 0).all())


@pytest.mark.parametrize("H", [20, 32])
def test_attention_large_logits_stay_finite(H):
    """Logits up to +-300 after scaling (exp(300) overflows fp32; the kernel's online softmax subtracts the running max):
    every output finite and within the same 5e-5 of each scale of float64 as at ordinary logits (measured on a B200: at
    most 9.1e-6)."""
    o, qt, cst, dc, scale = _attn_case(4099, H, seed=8 + H, logit=300.0)
    s = _attn_compare("attention large logits H=%d" % H, o, qt, cst, dc, scale, 5e-5)
    assert s.abs().max().item() >= 299.0 and s.min().item() < -100.0 and s.max().item() > 100.0


# ------------------------------------------------------------------------------------------------ E. GEMM at the c5 products
def _ref_atb(a_pair, b_pair, chunk=131072):
    """float64 A^T B of two [k, m] / [k, n] bf16 pairs (the operand values hi + lo the kernel multiplies), in row chunks."""
    k = a_pair[0].shape[0]
    out = torch.zeros(a_pair[0].shape[1], b_pair[0].shape[1], dtype=F64, device=DEV)
    for r0 in range(0, k, chunk):
        r1 = min(k, r0 + chunk)
        a = a_pair[0][r0:r1].double() + a_pair[1][r0:r1].double()
        b = b_pair[0][r0:r1].double() + b_pair[1][r0:r1].double()
        out.addmm_(a.t(), b)
    return out


def _split_rows(x32_fn, rows, cols, chunk=262144):
    hi = torch.empty(rows, cols, dtype=BF16, device=DEV)
    lo = torch.empty_like(hi)
    for i, r0 in enumerate(range(0, rows, chunk)):
        r1 = min(rows, r0 + chunk)
        h, l_ = native.split(x32_fn(r1 - r0, i))
        hi[r0:r1], lo[r0:r1] = h, l_
    return hi, lo


# The tensor cores accumulate each k-slice in fp32, and the error grows about in proportion to the rows of a slice: on a
# B200 the spatial dW_hh product (2 457 600 rows) measured 7.4e-3 of its scale as one slice, 1.5e-4 at the library's own
# split (about 50 000 rows per slice) and 4.8e-5 at 16 384 rows per slice.  The worst of the launches below measured
# 2.3e-4 (default) and 2.1e-4 (ordered), well past the 3e-5 of the smaller weight-gradient tests and within the 1e-3 the
# native pass is held to; the tolerance keeps a 2x margin over them.
C5_GEMM_TOL = 5e-4


def test_gemm_weight_gradients_of_the_c5_update_match_float64():
    """The grouped dW_hh and G^T [e | 1] launches of EdgeGruSequence.backward at T = 30, n = 4096, H = 20: A = column slices
    of the [rows, 1024] split image of G (row stride 1024), B = the split masked states / encoder rows [e | 1 | 0 x 7],
    split_k = 0, spatial (2 457 600 rows) and temporal (122 880 rows) problems in one launch.  Default and ordered mode
    against a float64 product of the same bf16 operand values within C5_GEMM_TOL of the scale."""
    T, n, H = 30, 4096, 20
    S = n * H
    TS, rows = T * S, T * (S + n)
    g_pair = _split_rows(lambda r, i: torch.randn(r, 1024, device=DEV, generator=_gen(100 + i)), rows, 1024)

    def masked(r, i):
        h = torch.randn(r, 256, device=DEV, generator=_gen(2000 + i)) * 0.5
        return h * (torch.rand(r, 1, device=DEV, generator=_gen(4000 + i)) > 0.03)
    hm_pair = _split_rows(masked, rows, 256)

    def enc(r, i):
        e = torch.zeros(r, 72, device=DEV)
        e[:, :64] = torch.relu(torch.randn(r, 64, device=DEV, generator=_gen(6000 + i)))
        e[:, 64] = 1.0
        return e
    e_pair = _split_rows(enc, rows, 72)
    sl = lambda p, r, c=slice(None): (p[0][r, c], p[1][r, c])
    sp, tp = slice(0, TS), slice(TS, rows)
    want = {"dW_hh spatial": _ref_atb(sl(g_pair, sp, slice(256, None)), sl(hm_pair, sp)),
            "dW_hh temporal": _ref_atb(sl(g_pair, tp, slice(256, None)), sl(hm_pair, tp)),
            "G^T[e|1] spatial": _ref_atb(sl(g_pair, sp), sl(e_pair, sp)),
            "G^T[e|1] temporal": _ref_atb(sl(g_pair, tp), sl(e_pair, tp))}
    errs = []
    for mode in ("default", "ordered"):
        dwh = torch.zeros(2, 768, 256, device=DEV)
        dwx = torch.zeros(2, 1024, 72, device=DEV)
        native.DETERMINISTIC = mode == "ordered"
        try:
            native.gemm([dict(a=sl(g_pair, sp, slice(256, None)), a_mn=True, b=sl(hm_pair, sp), b_mn=True, c=dwh[0], split_k=0),
                         dict(a=sl(g_pair, tp, slice(256, None)), a_mn=True, b=sl(hm_pair, tp), b_mn=True, c=dwh[1], split_k=0)])
            native.gemm([dict(a=sl(g_pair, sp), a_mn=True, b=sl(e_pair, sp), b_mn=True, c=dwx[0], split_k=0),
                         dict(a=sl(g_pair, tp), a_mn=True, b=sl(e_pair, tp), b_mn=True, c=dwx[1], split_k=0)])
        finally:
            native.DETERMINISTIC = False
        torch.cuda.synchronize()
        for name, got in (("dW_hh spatial", dwh[0]), ("dW_hh temporal", dwh[1]), ("G^T[e|1] spatial", dwx[0]),
                          ("G^T[e|1] temporal", dwx[1])):
            scale = want[name].abs().max().item()
            errs.append(("c5 %s (%s)" % (name, mode), (got.double() - want[name]).abs().max().item() / scale))
    for name, rel in errs:
        print("%-48s err %.2e of the scale (tol %.1e)" % (name, rel, C5_GEMM_TOL))
    assert not [e for e in errs if not e[1] <= C5_GEMM_TOL], errs


STRIDED_LAYOUTS = [(211, 3), (204, 4)]      # (row stride, first column): ldc % 8 != 0; the first also ldc % 4 != 0, C 4 B aligned


@pytest.mark.parametrize("ldw,col", STRIDED_LAYOUTS)
@pytest.mark.parametrize("mode", ["store", "accumulate", "atomic_split", "ordered_split"])
def test_gemm_into_a_strided_column_slice(ldw, col, mode):
    """C = wide[:, col:col + 200] with a row stride that is not a multiple of 8: the scalar epilogue of gemm_bf16x3_kernel,
    and for the ordered split-K the vec = 0 path of splitk_reduce_kernel (ldc % 4 != 0 or C not 16-byte aligned).  Against
    float64 within 3e-5 of the scale; every element of `wide` outside C keeps its NaN."""
    m, nn, k = 304, 200, 1000                 # m, n: operand leading dimensions (multiples of 8); 304 leaves a ragged tile
    dy, x = _randn(k, m, seed=70), _randn(k, nn, seed=71)
    wide = torch.full((m, ldw), float("nan"), device=DEV)
    c0 = _randn(m, nn, seed=72)
    c = wide[:, col:col + nn]
    want = dy.double().t() @ x.double()
    p = dict(a=native.split(dy), a_mn=True, b=native.split(x), b_mn=True, c=c)
    if mode != "store":
        c.copy_(c0)
        want = want + c0.double()
    if mode == "accumulate":
        p["accumulate"] = True
    elif mode.endswith("split"):
        p["split_k"] = 3
    native.DETERMINISTIC = mode == "ordered_split"
    try:
        if mode == "ordered_split":
            assert native.ordered_workspace([p])[1] == [3]
        native.gemm([p])
    finally:
        native.DETERMINISTIC = False
    torch.cuda.synchronize()
    _check("strided C ldc=%d col=%d %s" % (ldw, col, mode), c, want, 3e-5)
    outside = torch.cat([wide[:, :col].reshape(-1), wide[:, col + nn:].reshape(-1)])
    assert bool(outside.isnan().all()), "the product wrote outside its column slice"


# ------------------------------------------------------------------------------------------------ F. the native pass vs float64
def _benchmark_case(n, H, T):
    from crowdnav_dsrnn_b200.model import Policy
    from crowdnav_dsrnn_b200.spaces import crowd_spaces

    obs_space, act_space = crowd_spaces(H)
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        policy = Policy(obs_space.spaces, act_space, base="srnn", base_kwargs=Config(human_num=H)).to(DEV)
    g = torch.Generator(device=DEV).manual_seed(0)
    obs = {"robot_node": torch.randn(T * n, 1, 7, device=DEV, generator=g),
           "temporal_edges": torch.randn(T * n, 1, 2, device=DEV, generator=g),
           "spatial_edges": torch.randn(T * n, H, 2, device=DEV, generator=g) * 3}
    masks = (torch.rand(T * n, 1, device=DEV, generator=g) > 0.03).float()
    action = torch.randn(T * n, 2, device=DEV, generator=g)
    h0 = {"human_node_rnn": torch.randn(n, 1, 128, device=DEV, generator=g) * 0.3,
          "human_human_edge_rnn": torch.randn(n, H + 1, 256, device=DEV, generator=g) * 0.3}
    return policy, obs, masks, action, h0


def _full_pass(policy, obs, h0, masks, action, dtype):
    """evaluate_actions + backward of the loss sequence_impls_agree uses; returns outputs, final states, every parameter
    gradient and the gradient of h0 (all detached)."""
    cast = lambda t: t.to(dtype)
    policy.zero_grad(set_to_none=True)
    hx = {k: cast(v).clone().requires_grad_(True) for k, v in h0.items()}
    value, logp, _, out = policy.evaluate_actions({k: cast(v) for k, v in obs.items()}, dict(hx), cast(masks), cast(action))
    weights = torch.linspace(0, 1, value.numel(), device=DEV, dtype=dtype).view_as(value)
    ((value * weights).sum() + 0.3 * logp.sum() + 0.01 * out["human_human_edge_rnn"].sum()
     + 0.02 * out["human_node_rnn"].sum()).backward()
    res = {"value": value.detach(), "log_prob": logp.detach(), "h_edge": out["human_human_edge_rnn"].detach(),
           "h_node": out["human_node_rnn"].detach()}
    res.update({"grad h0 " + k: hx[k].grad.detach() for k in sorted(hx)})
    grads = {k: q.grad.detach().clone() for k, q in policy.named_parameters() if q.grad is not None}
    policy.zero_grad(set_to_none=True)
    return res, grads


# q . b_s adds the same constant to every logit of a sample, which the softmax ignores: the gradient of b_s is exactly zero,
# and what either graph returns for it is rounding noise.  It is held to 1e-3 of the gradient of the layer's weight.
ZERO_GRAD = "base.attn.spatial_edge_layer.0.bias"


def test_native_pass_at_the_benchmark_shape_matches_float64():
    """One native forward + backward at 4096 envs x 20 humans x T = 30 (the c5 update's pass), in default and in ordered
    mode, against the same policy cast to float64 with sequence_impl = "per_step": values, log-probs, final hidden states
    and the gradient of h0 within 1e-3 of max(1, scale), every parameter gradient within 1e-3 of its own scale -- the bar
    sequence_impls_agree holds the native path to at small shapes (worst measured on a B200: 4.0e-4, the edge GRUs' input
    weight gradients in default mode).  The float64 per-step graph (forward + backward) peaks at 82.1 GB on top of what is
    allocated before it (measured with torch.cuda.max_memory_allocated)."""
    n, H, T = 4096, 20, 30
    policy, obs, masks, action, h0 = _benchmark_case(n, H, T)
    ref_policy = copy.deepcopy(policy).double()
    ref_policy.sequence_impl = "per_step"
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    want, want_grads = _full_pass(ref_policy, obs, h0, masks, action, F64)
    torch.cuda.synchronize()
    print("float64 per-step pass at n=%d H=%d T=%d: peak %.1f GB above the %.1f GB held before it"
          % (n, H, T, (torch.cuda.max_memory_allocated() - base) / 1e9, base / 1e9))
    del ref_policy
    torch.cuda.empty_cache()
    policy.sequence_impl = "native"
    for mode in ("default", "ordered"):
        native.DETERMINISTIC = mode == "ordered"
        try:
            got, grads = _full_pass(policy, obs, h0, masks, action, torch.float32)
        finally:
            native.DETERMINISTIC = False
        for k in want:
            _check("c5 pass (%s) %s" % (mode, k), got[k], want[k], 1e-3)
        assert sorted(grads) == sorted(want_grads) and len(grads) >= 40
        bad = []
        for k in want_grads:
            scale = max(want_grads[k].abs().max().item(), 1e-3)
            if k == ZERO_GRAD:
                scale = want_grads[ZERO_GRAD.replace("bias", "weight")].abs().max().item()
            err = (grads[k].double() - want_grads[k]).abs().max().item()
            print("%-48s err %.3e of scale %.3e = %.2e (tol 1.0e-03)" % ("c5 pass (%s) grad %s" % (mode, k), err, scale, err / scale))
            if not err <= 1e-3 * scale:
                bad.append("%s: err %.3e scale %.3e" % (k, err, scale))
        assert not bad, (mode, bad)
