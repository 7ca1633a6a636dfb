"""Native building blocks of the PPO update (SURVEY.md 8(f) row N1): autograd Functions whose forward AND backward run on
the library's hand-written sm_100a kernels -- no cuBLAS product anywhere in `Policy.evaluate_actions` + `backward()`.

* `gemm`               cn_gemm_bf16x3: TMA-fed tcgen05 split-bf16 3-pass GEMM (csrc/gemm_bf16x3.cu), K-major or MN-major
                       operands, grouped problems, split-K with atomic accumulation for the weight gradients -- or, while
                       `ordered()` holds, cn_gemm_bf16x3_ordered: the split-K partial products summed in a fixed order.
* `linear`             y = act(x W^T + b) and its three backward products (dx = dy W, dW = dy^T x, db) on that kernel.
* `EdgeGruSequence`    the two edge GRUs of the DS-RNN over a [T, n] rollout chunk (srnn_model.py:53-104, 201-215): forward =
                       T launches of the rollout's tcgen05 edge kernel in training mode (cn_dsrnn_edge_sequence_step: also
                       writes the gate values and the split-bf16 operands of the backward); backward = per step one gate
                       kernel (cn_gru_gates_backward_pairs) + one grouped recurrent product, then the input and weight
                       gradients of the whole sequence as three grouped GEMM launches.

Reproducibility: the split-K weight gradients and the edge-encoder gradient combine partial sums from many CTAs.  By default
they do so with atomics, whose order varies from run to run (results agree to ~1e-6 relative, not bit for bit).  While
`ordered()` is true -- inside an update of `PPO(deterministic=True)` (training.cuda_deterministic), or whenever
`torch.use_deterministic_algorithms(True)` is in effect -- they write their partial sums to a workspace taken from torch's
caching allocator and add them in a fixed order instead, so the same inputs give the same gradients bit for bit.

Everything here needs CUDA tensors on a B200; there is no CPU fallback (the CPU tests exercise the torch restatement in
model.py, which is also the cross-check of these kernels on the GPU).
"""
import ctypes as C

import torch

from . import _lib, abi

BF16 = torch.bfloat16

# Set by PPO(deterministic=True) for the duration of its update (as PPO sets model.SEQUENCE_GEMM); see `ordered`.
DETERMINISTIC = False


def ordered():
    """True when reductions over many CTAs must be summed in a fixed order (bit-reproducible) rather than with atomics."""
    return DETERMINISTIC or torch.are_deterministic_algorithms_enabled()


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class _on_device(object):
    """Pointer-only entry points launch on the current device: switch to the tensors' device when it differs."""

    def __init__(self, device):
        self.ctx = None
        if device.index is not None and device.index != torch.cuda.current_device():
            self.ctx = torch.cuda.device(device)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)


def split(x):
    """fp32 tensor -> (hi, lo) bfloat16 tensors of the same shape with x ~= hi + lo to 2^-16 relative (cn_split_bf16)."""
    x = x.contiguous()
    if x.dtype is not torch.float32 or not x.is_cuda:
        raise _lib.CrowdNavLibraryError("native.split needs a CUDA float32 tensor")
    hi = torch.empty(x.shape, dtype=BF16, device=x.device)
    lo = torch.empty_like(hi)
    n = x.numel()
    if n == 0:
        return hi, lo
    if n % 4:
        raise _lib.CrowdNavLibraryError("native.split: element count must be a multiple of 4")
    with _on_device(x.device):
        _lib.check(_lib.load().cn_split_bf16(_ptr(x), _ptr(hi), _ptr(lo), n, _stream(x.device)), "cn_split_bf16")
    return hi, lo


def _operand(pair, mn_major):
    hi, lo = pair
    if hi.dim() != 2 or hi.dtype is not BF16 or (hi.shape[1] > 1 and hi.stride(1) != 1):
        raise ValueError("GEMM operands are 2-D bfloat16 matrices with unit column stride")
    ld = hi.stride(0) if hi.shape[0] > 1 else max(hi.stride(0), hi.shape[1])
    if lo is not None and (lo.shape != hi.shape or lo.stride() != hi.stride()):
        raise ValueError("hi and lo of a pair must have the same layout")
    return abi.CnGemmOperand(_ptr(hi), _ptr(lo), ld, 1 if mn_major else 0, 0)


def _gemm_array(problems):
    if not 1 <= len(problems) <= abi.GEMM_MAX_PROBLEMS:
        raise ValueError("1..%d problems per launch" % abi.GEMM_MAX_PROBLEMS)
    arr = (abi.CnGemm * len(problems))()
    keep = []
    dev = problems[0]["c"].device
    for g, p in zip(arr, problems):
        a_mn, b_mn = bool(p.get("a_mn", False)), bool(p.get("b_mn", False))
        a_hi, b_hi, c = p["a"][0], p["b"][0], p["c"]
        k, m = (a_hi.shape if a_mn else a_hi.shape[::-1])
        k2, n = (b_hi.shape if b_mn else b_hi.shape[::-1])
        if k != k2 or c.dim() != 2 or tuple(c.shape) != (m, n) or c.dtype is not torch.float32 or (n > 1 and c.stride(1) != 1):
            raise ValueError("inconsistent GEMM shapes: A %s (mn=%s) B %s (mn=%s) C %s" % (tuple(a_hi.shape), a_mn, tuple(b_hi.shape), b_mn, tuple(c.shape)))
        bias = p.get("bias")
        if bias is not None:
            bias = bias.contiguous()
            keep.append(bias)
        g.a, g.b = _operand(p["a"], a_mn), _operand(p["b"], b_mn)
        g.c, g.ldc, g.bias = _ptr(c), (c.stride(0) if m > 1 else max(c.stride(0), n)), _ptr(bias)
        g.m, g.n, g.k = m, n, k
        g.act, g.accumulate, g.split_k = int(p.get("act", 0)), int(bool(p.get("accumulate", False))), int(p.get("split_k", 1))
    return arr, keep, dev


def ordered_workspace(problems):
    """(bytes, slice count of each problem) of an ordered launch of `problems` (same dicts as `gemm`); host-side only."""
    arr, _, _ = _gemm_array(problems)
    need, slices = C.c_size_t(), (C.c_int * len(problems))()
    _lib.check(_lib.load().cn_gemm_bf16x3_ordered_workspace_bytes(arr, len(problems), C.byref(need), slices),
               "cn_gemm_bf16x3_ordered_workspace_bytes")
    return need.value, list(slices)


def gemm(problems):
    """Launch up to abi.GEMM_MAX_PROBLEMS products in one grouped tcgen05 kernel.  Each problem is a dict:
    a=(hi, lo), a_mn=bool, b=(hi, lo), b_mn=bool, c=fp32 [m, n] (unit column stride), bias=None, act=0, accumulate=False,
    split_k=1 (0 = library's choice; >1 / 0 add partial products to c: c must be initialised).  While `ordered()` holds the
    partial products are summed in slice order (cn_gemm_bf16x3_ordered, workspace from the caching allocator)."""
    arr, keep, dev = _gemm_array(problems)
    lib = _lib.load()
    with _on_device(dev):
        if ordered():
            need = C.c_size_t()
            _lib.check(lib.cn_gemm_bf16x3_ordered_workspace_bytes(arr, len(problems), C.byref(need), None),
                       "cn_gemm_bf16x3_ordered_workspace_bytes")
            ws = torch.empty(need.value, dtype=torch.uint8, device=dev) if need.value else None
            _lib.check(lib.cn_gemm_bf16x3_ordered(arr, len(problems), _ptr(ws), need.value, _stream(dev)), "cn_gemm_bf16x3_ordered")
        else:
            _lib.check(lib.cn_gemm_bf16x3(arr, len(problems), _stream(dev)), "cn_gemm_bf16x3")
    COUNTERS["gemm_launches"] += 1


def encoder_grad(de, e_hi, ld_e, x, dw, db):
    """dw [64, 2] += sum_rows [e > 0] de x^T, db [64] += sum_rows [e > 0] de (cn_encoder_grad; cn_encoder_grad_ordered while
    `ordered()` holds).  de [rows, 64] fp32, e_hi the bf16 image of e with row stride ld_e, x [rows, 2]."""
    lib, dev, rows = _lib.load(), de.device, x.shape[0]
    with _on_device(dev):
        if ordered():
            ws = torch.empty(lib.cn_encoder_grad_ordered_workspace_bytes(rows), dtype=torch.uint8, device=dev)
            _lib.check(lib.cn_encoder_grad_ordered(_ptr(de), _ptr(e_hi), ld_e, _ptr(x), _ptr(dw), _ptr(db), rows, _ptr(ws), ws.numel(),
                                                   _stream(dev)), "cn_encoder_grad_ordered")
        else:
            _lib.check(lib.cn_encoder_grad(_ptr(de), _ptr(e_hi), ld_e, _ptr(x), _ptr(dw), _ptr(db), rows, _stream(dev)), "cn_encoder_grad")


COUNTERS = {"gemm_launches": 0, "kernel_launches": 0}
ACT = {None: 0, "relu": 1, "tanh": 2}


def _native_ok(x, w):
    return x.is_cuda and x.dtype is torch.float32 and w.shape[1] % 8 == 0 and w.shape[0] % 8 == 0 and x.shape[0] > 0


class _Linear(torch.autograd.Function):
    """y = act(x W^T + b) with x [M, K], W [N, K]: forward, dx, dW on cn_gemm_bf16x3; db / the activation derivative in torch."""

    @staticmethod
    def forward(ctx, x, w, b, act):
        xp, wp = split(x), split(w)
        y = torch.empty(x.shape[0], w.shape[0], dtype=torch.float32, device=x.device)
        gemm([dict(a=xp, b=wp, c=y, bias=b, act=act)])
        ctx.act = act
        ctx.has_bias = b is not None
        ctx.save_for_backward(xp[0], xp[1], wp[0], wp[1], y if act else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x_hi, x_lo, w_hi, w_lo, y = ctx.saved_tensors
        if ctx.act == 1:
            dy = dy * (y > 0)
        elif ctx.act == 2:
            dy = torch.addcmul(dy, dy * y, y, value=-1.0)           # dy (1 - y^2)
        dy = dy.contiguous()
        dyp = split(dy)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty(x_hi.shape, dtype=torch.float32, device=dy.device)
            gemm([dict(a=dyp, b=(w_hi, w_lo), b_mn=True, c=dx)])                      # [M, N] x [N, K]
        if ctx.needs_input_grad[1]:
            dw = torch.zeros(w_hi.shape, dtype=torch.float32, device=dy.device)
            gemm([dict(a=dyp, a_mn=True, b=(x_hi, x_lo), b_mn=True, c=dw, split_k=0)])  # [N, M] x [M, K], reduction over the rows
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy.sum(0)
        return dx, dw, db, None


def linear(x, module, act=None):
    """`act(module(x))` for an nn.Linear on the native GEMM; x [..., K]."""
    w, b = module.weight, module.bias
    lead = x.shape[:-1]
    x2 = x.reshape(-1, x.shape[-1])
    if not _native_ok(x2, w):
        y = torch.nn.functional.linear(x, w, b)
        return torch.relu(y) if act == "relu" else torch.tanh(y) if act == "tanh" else y
    return _Linear.apply(x2, w, b, ACT[act]).view(*lead, w.shape[0])


def matmul_nt(x, w):
    """x [M, K] @ w[N, K]^T without bias (w need not be a parameter)."""
    if not _native_ok(x, w):
        return x @ w.t()
    return _Linear.apply(x, w, None, 0)


# ---------------------------------------------------------------------------------------------------------------------
class AttentionMix(torch.autograd.Function):
    """c = sum_i softmax_i((o_i . qt + cst) * scale) o_i over a batch (srnn_model.py:256-339 with the key projection folded
    into the query); forward and backward are one HBM-bound pass over o each (csrc/dsrnn_train.cu)."""

    @staticmethod
    def forward(ctx, o, qt, cst, scale):
        o, qt, cst = o.contiguous(), qt.contiguous(), cst.contiguous()
        B, H = o.shape[0], o.shape[1]
        c = torch.empty(B, 256, dtype=torch.float32, device=o.device)
        alpha = torch.empty(B, H, dtype=torch.float32, device=o.device)
        with _on_device(o.device):
            _lib.check(_lib.load().cn_attention_train_forward(_ptr(o), _ptr(qt), _ptr(cst), _ptr(c), _ptr(alpha), float(scale), B, H,
                                                              _stream(o.device)), "cn_attention_train_forward")
        COUNTERS["kernel_launches"] += 1
        ctx.scale = float(scale)
        ctx.save_for_backward(o, qt, alpha)
        return c

    @staticmethod
    def backward(ctx, dc):
        o, qt, alpha = ctx.saved_tensors
        B, H = o.shape[0], o.shape[1]
        dc = dc.contiguous()
        d_o, d_qt = torch.empty_like(o), torch.empty_like(qt)
        d_cst = torch.empty(B, dtype=torch.float32, device=o.device)
        with _on_device(o.device):
            _lib.check(_lib.load().cn_attention_train_backward(_ptr(o), _ptr(qt), _ptr(alpha), _ptr(dc), _ptr(d_o), _ptr(d_qt), _ptr(d_cst),
                                                               ctx.scale, B, H, _stream(o.device)), "cn_attention_train_backward")
        COUNTERS["kernel_launches"] += 1
        return d_o, d_qt, d_cst, None


# ---------------------------------------------------------------------------------------------------------------------
class EdgeGruSequence(torch.autograd.Function):
    """Both edge GRUs of the DS-RNN over a [T, n] chunk.

    forward(policy, se [T, S, 2], te [T, n, 2], h0 [S + n, 256] (spatial rows, then temporal rows), masks [T, n],
            12 parameters) -> (o_s [T*S, 256], o_t [T*n, 256]): the two halves of ONE buffer in the sequence layout (spatial
            rows of all steps, then temporal rows), returned separately so that their gradients arrive separately.
    """

    @staticmethod
    def forward(ctx, policy, se, te, h0, masks, s_enc_w, s_enc_b, s_w_ih, s_w_hh, s_b_ih, s_b_hh,
                t_enc_w, t_enc_b, t_w_ih, t_w_hh, t_b_ih, t_b_hh):
        dev = se.device
        T, S = se.shape[0], se.shape[1]
        n = te.shape[1]
        H = S // n
        lib = policy._ensure_handle(dev)         # packs the CURRENT weights (bf16 hi/lo images) if they changed
        rows = T * (S + n)
        f32 = dict(dtype=torch.float32, device=dev)
        hs = torch.empty(rows, 256, **f32)
        ws = torch.empty(rows, 1024, **f32)
        hm_hi, hm_lo = torch.empty(rows, 256, dtype=BF16, device=dev), torch.empty(rows, 256, dtype=BF16, device=dev)
        e_hi, e_lo = torch.empty(rows, 72, dtype=BF16, device=dev), torch.empty(rows, 72, dtype=BF16, device=dev)   # [e | 1 | 0 x 7]
        se, te, h0, masks = se.contiguous(), te.contiguous(), h0.contiguous(), masks.contiguous()
        stream = _stream(dev)
        io = abi.CnEdgeSeqStep()
        io.h_out, io.ws, io.hm_hi, io.hm_lo, io.e_hi, io.e_lo = _ptr(hs), _ptr(ws), _ptr(hm_hi), _ptr(hm_lo), _ptr(e_hi), _ptr(e_lo)
        for t in range(T):
            io.temporal_edges, io.spatial_edges, io.masks = _ptr(te[t]), _ptr(se[t]), _ptr(masks[t])
            if t == 0:
                io.h_in, io.in_row_spatial, io.in_row_temporal = _ptr(h0), 0, S
            else:
                io.h_in, io.in_row_spatial, io.in_row_temporal = _ptr(hs), (t - 1) * S, T * S + (t - 1) * n
            io.out_row_spatial, io.out_row_temporal = t * S, T * S + t * n
            _lib.check(lib.cn_dsrnn_edge_sequence_step(policy._handle, n, H, C.byref(io), stream), "cn_dsrnn_edge_sequence_step")
        COUNTERS["kernel_launches"] += T
        ctx.dims = (T, S, n, H)
        ctx.save_for_backward(se, te, h0, masks, hs, ws, hm_hi, hm_lo, e_hi, e_lo, s_w_ih, s_w_hh, t_w_ih, t_w_hh)
        return hs[:T * S], hs[T * S:]

    @staticmethod
    def backward(ctx, grad_os, grad_ot):
        se, te, h0, masks, hs, ws, hm_hi, hm_lo, e_hi, e_lo, s_w_ih, s_w_hh, t_w_ih, t_w_hh = ctx.saved_tensors
        T, S, n, H = ctx.dims
        dev = hs.device
        lib = _lib.load()
        stream = _stream(dev)
        rows = T * (S + n)
        TS = T * S
        zeros = lambda r: torch.zeros(r, 256, dtype=torch.float32, device=dev)
        grad_seg = ((zeros(TS) if grad_os is None else grad_os.contiguous()), (zeros(rows - TS) if grad_ot is None else grad_ot.contiguous()))
        g_hi = torch.empty(rows, 1024, dtype=BF16, device=dev)
        g_lo = torch.empty(rows, 1024, dtype=BF16, device=dev)
        d = torch.empty(S + n, 256, dtype=torch.float32, device=dev)        # dL/d(masked state of the step), spatial | temporal rows
        m_sp = masks.view(T, n, 1).expand(T, n, H).reshape(T, S).contiguous()   # per-row masks of the spatial rows
        whh_s, whh_t = split(s_w_hh), split(t_w_hh)                         # [768, 256] = [K, N]: MN-major B of d += G[:, 256:] W_hh
        # (first row in the sequence layout, first row in d / h0, rows per step, masks, W_hh, incoming gradient)
        seg = ((0, 0, S, m_sp, whh_s, grad_seg[0]), (TS, S, n, masks, whh_t, grad_seg[1]))
        for t in range(T - 1, -1, -1):
            probs = []
            live = 1 if t + 1 < T else 0
            for base, doff, R, mk, whh, gseg in seg:
                lo_, hi_ = base + t * R, base + (t + 1) * R
                hprev = h0[doff:doff + R] if t == 0 else hs[lo_ - R:lo_]
                dseg = d[doff:doff + R]
                _lib.check(lib.cn_gru_gates_backward_pairs(_ptr(gseg[t * R:(t + 1) * R]), _ptr(dseg), live, _ptr(mk[t + 1]) if live else None,
                                                           _ptr(ws[lo_:hi_]), _ptr(hprev), _ptr(mk[t]), _ptr(g_hi[lo_:hi_]),
                                                           _ptr(g_lo[lo_:hi_]), R, 256, stream), "cn_gru_gates_backward_pairs")
                probs.append(dict(a=(g_hi[lo_:hi_, 256:], g_lo[lo_:hi_, 256:]), b=whh, b_mn=True, c=dseg, accumulate=True))
            gemm(probs)
        COUNTERS["kernel_launches"] += 2 * T
        grad_h0 = None
        if ctx.needs_input_grad[3]:
            grad_h0 = d * torch.cat([m_sp[0], masks[0]]).unsqueeze(1)
        # ---- whole-sequence products: encoder-side input gradient, weight gradients (reduction over all T*R rows)
        gs, gt = (g_hi[:TS], g_lo[:TS]), (g_hi[TS:], g_lo[TS:])
        perm = lambda w: torch.cat([w[512:], w[:512]], 0)                    # gate rows n | r | z: the column order of G[:, :768]
        de = torch.empty(rows, 64, dtype=torch.float32, device=dev)
        gemm([dict(a=(gs[0][:, :768], gs[1][:, :768]), b=split(perm(s_w_ih)), b_mn=True, c=de[:TS]),
              dict(a=(gt[0][:, :768], gt[1][:, :768]), b=split(perm(t_w_ih)), b_mn=True, c=de[TS:])])
        dwh = torch.zeros(2, 768, 256, dtype=torch.float32, device=dev)      # dW_hh
        dwx = torch.zeros(2, 1024, 72, dtype=torch.float32, device=dev)      # G^T [e | 1]: [:, :768, :64] dW_ih (rows n|r|z), [:, :, 64] column sums of G
        gemm([dict(a=(gs[0][:, 256:], gs[1][:, 256:]), a_mn=True, b=(hm_hi[:TS], hm_lo[:TS]), b_mn=True, c=dwh[0], split_k=0),
              dict(a=(gt[0][:, 256:], gt[1][:, 256:]), a_mn=True, b=(hm_hi[TS:], hm_lo[TS:]), b_mn=True, c=dwh[1], split_k=0)])
        gemm([dict(a=gs, a_mn=True, b=(e_hi[:TS], e_lo[:TS]), b_mn=True, c=dwx[0], split_k=0),
              dict(a=gt, a_mn=True, b=(e_hi[TS:], e_lo[TS:]), b_mn=True, c=dwx[1], split_k=0)])
        unperm = lambda w: torch.cat([w[256:], w[:256]], 0)                  # n | r | z -> r | z | n
        grads = []
        for k, (x, sl) in enumerate(((se.view(TS, 2), slice(0, TS)), (te.view(T * n, 2), slice(TS, rows)))):
            colsum = dwx[k, :, 64]                                           # [1024]: sums of pn | pr | pz | pn*r over all rows
            db_ih = torch.cat([colsum[256:768], colsum[:256]])
            db_hh = colsum[256:]
            dw_enc, db_enc = torch.zeros(64, 2, dtype=torch.float32, device=dev), torch.zeros(64, dtype=torch.float32, device=dev)
            encoder_grad(de[sl], e_hi[sl], 72, x, dw_enc, db_enc)            # ReLU mask + the two reductions in one pass over de
            grads.append((dw_enc, db_enc, unperm(dwx[k, :768, :64]), dwh[k], db_ih, db_hh))
        return (None, None, None, grad_h0, None) + grads[0] + grads[1]
