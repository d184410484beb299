"""Autograd bindings of kernel family 5 (csrc/policy_kernels.cu) plus the small amount of torch glue around them.

Only plain dense layers go through library GEMMs (torch.addmm / torch.mm -> cuBLAS); everything pairwise, sparse or
pointwise is one of our kernels.  fp32 throughout (parity mode: TF32 is switched off for the GEMMs by the caller).
"""
import collections
import ctypes

import torch

from . import _lib


def _L():
    return _lib.lib()


class GraphBatch:
    """Inputs of the DHGN encoder for S samples (a sample = one env at one time step).

    p [S,N,4] f32, e [S,4] f32, oxy [Bo,O,2] f32 (obstacle cells per map row), o_index [S] i32, o_count [Bo] i32,
    p_adj_bits [S,N,NW] i32, e_adj [S,N] u8, o_adj_bits [S,N,OW] i32."""

    def __init__(self, p, e, oxy, o_index, o_count, p_adj_bits, e_adj, o_adj_bits):
        self.p, self.e, self.oxy, self.o_index, self.o_count = p, e, oxy, o_index, o_count
        self.p_adj_bits, self.e_adj, self.o_adj_bits = p_adj_bits, e_adj, o_adj_bits
        self.S, self.N = p.shape[0], p.shape[1]
        self.O = oxy.shape[1]
        for t in (p, e, oxy, o_index, o_count, p_adj_bits, e_adj, o_adj_bits):
            assert t.is_contiguous() and t.is_cuda
        assert p.dtype == torch.float32 and e.dtype == torch.float32 and oxy.dtype == torch.float32
        assert o_index.dtype == torch.int32 and o_count.dtype == torch.int32 and e_adj.dtype == torch.uint8

    def _args(self, E, all_ones):
        P = _lib.ptr
        return (self.S, self.N, self.O, E, P(self.p), P(self.e), P(self.oxy), P(self.o_index), P(self.o_count),
                P(self.p_adj_bits), P(self.e_adj), P(self.o_adj_bits), 1 if all_ones else 0)


def pack_bits(dense):
    """float/bool 0-1 tensor [..., K] -> int32 words [..., ceil(K/32)] (bit k&31 of word k>>5)."""
    K = dense.shape[-1]
    KW = (K + 31) // 32
    b = (dense != 0)
    if KW * 32 != K:
        b = torch.nn.functional.pad(b, (0, KW * 32 - K))
    b = b.reshape(*dense.shape[:-1], KW, 32).to(torch.int64)
    w = (b << torch.arange(32, device=dense.device, dtype=torch.int64)).sum(-1)
    w = torch.where(w >= 2 ** 31, w - 2 ** 32, w)
    return w.to(torch.int32).contiguous()


# ---------------------------------------------------------------------------------------------------- dense layers
USE_TENSOR_CORES = True    # 3xTF32 tcgen05 GEMM for the E-wide layers (fp32-level accuracy); False -> library sgemm


def _tc_ok(x, W, x2):
    N, K = W.shape
    K1 = x.shape[1]
    return (USE_TENSOR_CORES and x.is_cuda and x.dtype == torch.float32 and N % 128 == 0 and K1 % 32 == 0
            and (K - K1) % 32 == 0 and W.stride(1) == 1 and W.stride(0) % 4 == 0 and W.data_ptr() % 16 == 0)


USE_ROWGEMM = True          # persistent row-tile kernel (csrc/rowgemm_tf32x3.cu) when N, K1, K2 are multiples of 128
ROWGEMM_MIN_ROWS = 256      # below: the tile-per-CTA kernel (a performance threshold only; tests lower both to exercise the
WGRAD_MIN_ROWS = 2048       # production kernels on small fixtures)
CALLS = collections.Counter()   # launches per tensor-core kernel family (tests assert the production path really ran)
_PACK_CACHE = {}
_PACK_SCOPE = [0]


class pack_scope:
    """Within the scope, packed (hi/lo split, swizzled) weight images are cached per weight view: the weights must not change
    inside it (MAPPO.train: one optimizer step per epoch, after all minibatches)."""

    def __enter__(self):
        _PACK_SCOPE[0] += 1
        return self

    def __exit__(self, *exc):
        _PACK_SCOPE[0] -= 1
        if _PACK_SCOPE[0] == 0:
            _PACK_CACHE.clear()
        return False


def _packed_weight(W, N, K, stride_n, stride_k):
    """Packed image of B[n][k] = W.data[n*stride_n + k*stride_k] (n < N, k < K)."""
    key = (W.data_ptr(), N, K, stride_n, stride_k, torch.cuda.current_stream().cuda_stream)   # packed on the stream that uses it
    if _PACK_SCOPE[0] and key in _PACK_CACHE:
        return _PACK_CACHE[key]
    nbytes = int(_L().marl_rowgemm_pack_bytes(N, K))
    buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=W.device)
    off = (-buf.data_ptr()) % 1024
    packed = buf[off:off + nbytes]
    _lib.check(_L().marl_rowgemm_pack(W.data_ptr(), stride_n, stride_k, N, K, packed.data_ptr(), _lib.stream_ptr()), "marl_rowgemm_pack")
    if _PACK_SCOPE[0]:
        _PACK_CACHE[key] = packed
    return packed


def _rowgemm_ok(M, N, K1, K2):
    return USE_ROWGEMM and N % 128 == 0 and N <= 512 and K1 % 128 == 0 and K2 % 128 == 0 and M >= ROWGEMM_MIN_ROWS


def _aligned_rows(t):
    return t if (t.stride(1) == 1 and t.stride(0) % 4 == 0 and t.data_ptr() % 16 == 0) else t.contiguous()


def _tc_t_ok(dy, Wslice):
    """dX = dY Wslice on the tensor cores: reduction over Wslice.shape[0] (must equal dy.shape[1]), output width Wslice.shape[1]."""
    N, K = Wslice.shape
    return (USE_TENSOR_CORES and dy.is_cuda and dy.dtype == torch.float32 and K % 128 == 0 and N % 32 == 0 and Wslice.stride(1) == 1
            and Wslice.data_ptr() % 16 == 0 and Wslice.stride(0) % 4 == 0)


def _gemm_tc(x, x2, W, bias, add, relu, out=None, transposed=False):
    """C = act(x B[:, :K1]^T + x2 B[:, K1:]^T + bias + add), B = W (nn.Linear weight [N,K]) or, with transposed=True, W^T
    (then W is [K, N]: dX = dY W without materialising the transpose)."""
    M, K1 = x.shape
    if transposed:
        K, N = W.shape
        stride_n, stride_k = W.stride(1), W.stride(0)
    else:
        N, K = W.shape
        stride_n, stride_k = W.stride(0), W.stride(1)
    K2 = K - K1
    x = _aligned_rows(x)
    if x2 is not None:
        x2 = _aligned_rows(x2)
    if add is not None:
        add = _aligned_rows(add)
    if out is None:
        out = torch.empty(M, N, dtype=torch.float32, device=x.device)
    if _rowgemm_ok(M, N, K1, K2):
        packed = _packed_weight(W, N, K, stride_n, stride_k)
        CALLS["rowgemm"] += 1
        _lib.check(_L().marl_rowgemm_tf32x3(
            M, N, K1, K2, x.data_ptr(), x.stride(0), x2.data_ptr() if x2 is not None else None, x2.stride(0) if x2 is not None else 0,
            packed.data_ptr(), bias.data_ptr() if bias is not None else None, add.data_ptr() if add is not None else None,
            add.stride(0) if add is not None else 0, out.data_ptr(), out.stride(0), 1 if relu else 0, _lib.stream_ptr()),
            "marl_rowgemm_tf32x3")
        return out
    if transposed:
        W = W.t().contiguous()
    CALLS["gemm_tile"] += 1
    _lib.check(_L().marl_gemm_tf32x3(
        M, N, K1, K - K1, x.data_ptr(), x.stride(0), x2.data_ptr() if x2 is not None else None,
        x2.stride(0) if x2 is not None else 0, W.data_ptr(), W.stride(0), bias.data_ptr() if bias is not None else None,
        add.data_ptr() if add is not None else None, add.stride(0) if add is not None else 0, out.data_ptr(), N,
        1 if relu else 0, _lib.stream_ptr()), "marl_gemm_tf32x3")
    return out


def _wgrad_ok(dy, x):
    return (USE_TENSOR_CORES and dy.is_cuda and dy.dtype == torch.float32 and x.dtype == torch.float32 and dy.shape[0] >= WGRAD_MIN_ROWS
            and dy.shape[1] % 128 == 0 and x.shape[1] % 128 == 0 and dy.stride(1) == 1 and x.stride(1) == 1)


def wgrad(dy, x, out=None, col0=0, dbias=None):
    """dW = dy^T @ x on the tensor cores (3xTF32, deterministic split-K); writes into out[:, col0 : col0 + x.shape[1]] if given.
    dbias (a [N] tensor) additionally receives dy.sum(0), computed by the same kernel from the same loads."""
    R, N = dy.shape
    K = x.shape[1]
    if out is None:
        out = torch.empty(N, K, dtype=torch.float32, device=dy.device)
    if not _wgrad_ok(dy, x):
        CALLS["wgrad_library"] += 1
        out[:, col0:col0 + K] = dy.t() @ x
        if dbias is not None:
            dbias.copy_(dy.sum(0))
        return out
    ws = torch.empty(int(_L().marl_wgrad_workspace_bytes(R, N, K)), dtype=torch.uint8, device=dy.device)
    dst = out[:, col0:]
    CALLS["wgrad"] += 1
    _lib.check(_L().marl_wgrad_tf32x3(R, N, K, dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0), dst.data_ptr(), out.stride(0),
                                      dbias.data_ptr() if dbias is not None else None, 0, ws.data_ptr(), _lib.stream_ptr()),
               "marl_wgrad_tf32x3")
    return out


def relu_bwd(dy, out):
    """dy * (out > 0) in one pass (backward of a ReLU fused into a GEMM epilogue)."""
    if dy.numel() % 4 or not out.is_contiguous() or dy.data_ptr() % 16 or out.data_ptr() % 16:
        return dy * (out > 0)
    dst = torch.empty_like(dy)
    _lib.check(_L().marl_relu_bwd(dy.numel(), dy.data_ptr(), out.data_ptr(), dst.data_ptr(), _lib.stream_ptr()), "marl_relu_bwd")
    return dst


class _SkinnyLinear(torch.autograd.Function):
    """bias + p @ W4^T for a 4- or 8-wide input that needs no gradient (the pursuer-state part of the semantic layer,
    DHGN/mappo_parallel.py:286,303).  Backward: weight and bias gradients in ONE pass over dY (marl_skinny_wgrad) instead of a
    [K, R] x [R, E] library GEMM (a 1 ms SIMT sgemm at R = 492 K) plus a column-sum kernel."""

    @staticmethod
    def forward(ctx, p, W4, bias):
        ctx.save_for_backward(p)
        ctx.shape = (W4.shape[0], W4.shape[1])
        return torch.addmm(bias, p, W4.t())

    @staticmethod
    def backward(ctx, dy):
        (p,) = ctx.saved_tensors
        N, K = ctx.shape
        dy = dy.contiguous()
        R = dy.shape[0]
        dW = torch.empty(N, K, dtype=torch.float32, device=dy.device)
        db = torch.empty(N, dtype=torch.float32, device=dy.device)
        ws = torch.empty(int(_L().marl_skinny_wgrad_workspace_bytes(R, N, K)), dtype=torch.uint8, device=dy.device)
        _lib.check(_L().marl_skinny_wgrad(R, N, K, dy.data_ptr(), dy.stride(0), p.data_ptr(), p.stride(0), dW.data_ptr(), dW.stride(0),
                                          db.data_ptr(), ws.data_ptr(), _lib.stream_ptr()), "marl_skinny_wgrad")
        return None, dW, db


def skinny_outer(y, p):
    """y^T @ p for y [R, N], p [R, K <= 16] (row-major): [N, K], deterministic, one pass over y."""
    R, N = y.shape
    K = p.shape[1]
    if not (y.is_cuda and y.dtype == torch.float32 and p.dtype == torch.float32 and K <= 16 and y.stride(1) == 1 and p.stride(1) == 1):
        return y.t() @ p
    out = torch.empty(N, K, dtype=torch.float32, device=y.device)
    ws = torch.empty(int(_L().marl_skinny_wgrad_workspace_bytes(R, N, K)), dtype=torch.uint8, device=y.device)
    _lib.check(_L().marl_skinny_wgrad(R, N, K, y.data_ptr(), y.stride(0), p.data_ptr(), p.stride(0), out.data_ptr(), out.stride(0),
                                      None, ws.data_ptr(), _lib.stream_ptr()), "marl_skinny_wgrad")
    return out


def skinny_linear(p, W4, bias):
    """bias + p @ W4^T, p [R, 4 or 8] (data, no gradient), W4 [E, K] (may be a column slice of a wider weight)."""
    if p.is_cuda and p.dtype == torch.float32 and p.dim() == 2 and p.shape[1] in (4, 8) and p.stride(1) == 1 and not p.requires_grad:
        return _SkinnyLinear.apply(p, W4, bias)
    return torch.addmm(bias, p, W4.t())


class _LinearTC(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, x2, W, bias, add, relu):
        out = _gemm_tc(x, x2, W, bias, add, relu)
        ctx.relu = relu
        ctx.has = (x2 is not None, bias is not None, add is not None)
        ctx.save_for_backward(x, x2, W, out if relu else None)
        return out

    @staticmethod
    def backward(ctx, dy):
        x, x2, W, out = ctx.saved_tensors
        has_x2, has_bias, has_add = ctx.has
        dy = dy.contiguous()
        if ctx.relu:
            dy = relu_bwd(dy, out)
        K1 = x.shape[1]
        need = ctx.needs_input_grad
        dx = dx2 = dW = db = dadd = None
        if need[0]:   # dX = dY W[:, :K1]: same kernel, the weight slice packed through its transposed view
            dx = _gemm_tc(dy, None, W[:, :K1], None, None, False, transposed=True) if _tc_t_ok(dy, W[:, :K1]) else dy @ W[:, :K1]
        if has_x2 and need[1]:
            dx2 = _gemm_tc(dy, None, W[:, K1:], None, None, False, transposed=True) if _tc_t_ok(dy, W[:, K1:]) else dy @ W[:, K1:]
        want_db = has_bias and need[3]
        if want_db:
            db = torch.empty(W.shape[0], dtype=torch.float32, device=dy.device)
        if need[2]:   # weight gradient: reduction over the (huge) row dimension -> split-K tensor-core kernel (+ fused bias gradient)
            if has_x2:
                dW = torch.empty(W.shape[0], W.shape[1], dtype=torch.float32, device=dy.device)
                wgrad(dy, x, dW, 0, dbias=db if want_db else None)
                wgrad(dy, x2, dW, K1)
            else:
                dW = wgrad(dy, x, dbias=db if want_db else None)
        elif want_db:
            db = dy.sum(0)
        if has_add and need[4]:
            dadd = dy
        return dx, dx2, dW, db, dadd, None


def linear(x, W, bias=None, relu=False, x2=None, add=None):
    """act(cat([x, x2], 1) @ W.T + bias + add) for 2-D x; tensor-core path when the shape allows, library GEMM otherwise."""
    if _tc_ok(x, W, x2):
        return _LinearTC.apply(x, x2, W, bias, add, relu)
    CALLS["linear_library"] += 1
    xin = x if x2 is None else torch.cat([x, x2], dim=1)
    out = torch.addmm(bias, xin, W.t()) if bias is not None else xin @ W.t()
    if add is not None:
        out = out + add
    return torch.relu(out) if relu else out


class _MessageAgg(torch.autograd.Function):
    @staticmethod
    def forward(ctx, graph, all_ones, W0, b0, W1, b1, W2, b2):
        E = W0.shape[0]
        ws = [t.contiguous() for t in (W0, b0, W1, b1, W2, b2)]
        agg = torch.empty(graph.S, graph.N, 3, E, dtype=torch.float32, device=W0.device)
        _lib.check(_L().marl_dhgn_message_fwd(*graph._args(E, all_ones), *[_lib.ptr(t) for t in ws], _lib.ptr(agg),
                                              _lib.stream_ptr()), "marl_dhgn_message_fwd")
        ctx.graph, ctx.all_ones = graph, all_ones
        ctx.save_for_backward(*ws)
        return agg

    @staticmethod
    def backward(ctx, d_agg):
        ws = ctx.saved_tensors
        E = ws[0].shape[0]
        g = ctx.graph
        grads = [torch.zeros_like(t) for t in ws]
        # fixed-order reduction (bit-reproducible gradients); the workspace comes from the caching allocator on this stream, so
        # the actor / critic streams of concurrent minibatches never share one
        part = torch.empty(int(_L().marl_dhgn_message_bwd_workspace_bytes(g.N, g.O, E)), dtype=torch.uint8, device=d_agg.device)
        _lib.check(_L().marl_dhgn_message_bwd_det(*g._args(E, ctx.all_ones), *[_lib.ptr(t) for t in ws],
                                                  _lib.ptr(d_agg.contiguous()), *[_lib.ptr(t) for t in grads], _lib.ptr(part),
                                                  _lib.stream_ptr()), "marl_dhgn_message_bwd_det")
        return (None, None, *grads)


def message_agg(graph, all_ones, W0, b0, W1, b1, W2, b2):
    """[S,N,3,E]: mean-aggregated ReLU messages of the three relations (input of AGG_vertex_0)."""
    return _MessageAgg.apply(graph, all_ones, W0, b0, W1, b1, W2, b2)


def fcra_agg(hist, p_adj_bits, all_ones, S, N, E, sample_stride=None, agent_stride=None):
    """L1norm(adj) @ hist (no gradient: history embeddings are data).  hist: tensor whose element (s,j,:) lives at
    data_ptr + (s*sample_stride + j*agent_stride)*4 bytes (defaults: contiguous [S,N,E])."""
    out = torch.empty(S, N, E, dtype=torch.float32, device=hist.device)
    ss = N * E if sample_stride is None else sample_stride
    as_ = E if agent_stride is None else agent_stride
    _lib.check(_L().marl_fcra_agg(S, N, E, hist.data_ptr(), ss, as_, _lib.ptr(p_adj_bits), 1 if all_ones else 0,
                                  _lib.ptr(out), _lib.stream_ptr()), "marl_fcra_agg")
    return out


USE_GRU_SEQ = True         # hidden size 128: the recurrence runs as one persistent kernel per direction (csrc/gru_seq.cu)


def _gru_pack(w_hh):
    """Pre-split / pre-swizzled images of W_hh for marl_gru_seq_{fwd,bwd} (1024-byte aligned)."""
    nbytes = int(_L().marl_gru_pack_bytes())
    buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=w_hh.device)
    off = (-buf.data_ptr()) % 1024
    packed = buf[off:off + nbytes]
    _lib.check(_L().marl_gru_pack(w_hh.detach().contiguous().data_ptr(), packed.data_ptr(), _lib.stream_ptr()), "marl_gru_pack")
    return packed


class _GRULayer(torch.autograd.Function):
    """One nn.GRU layer over a whole sequence: the input projection is one GEMM over all steps, the recurrence is
    one [R,E]x[E,3E] GEMM + one fused cell kernel per step."""

    @staticmethod
    def forward(ctx, x, h0, w_ih, w_hh, b_ih, b_hh):
        T, R, E = x.shape
        need = any(ctx.needs_input_grad)
        x = x.contiguous()
        tc = _tc_ok(x.view(T * R, E), w_ih, None) and _tc_ok(x.view(T * R, E), w_hh, None)
        if tc:
            gi_all = _gemm_tc(x.view(T * R, E), None, w_ih, b_ih, None, False).view(T, R, 3 * E)
        else:
            gi_all = torch.addmm(b_ih, x.view(T * R, E), w_ih.t()).view(T, R, 3 * E)
        out = torch.empty(T, R, E, dtype=x.dtype, device=x.device)
        saves = torch.empty(4, T, R, E, dtype=x.dtype, device=x.device) if need else None
        if tc and E == 128 and USE_GRU_SEQ:
            # whole recurrence in one persistent kernel (csrc/gru_seq.cu)
            packed = _gru_pack(w_hh)
            CALLS["gru_seq_fwd"] += 1
            _lib.check(_L().marl_gru_seq_fwd(T, R, E, gi_all.data_ptr(), h0.contiguous().data_ptr(), packed.data_ptr(),
                                             b_hh.contiguous().data_ptr(), out.data_ptr(), saves.data_ptr() if need else None,
                                             _lib.stream_ptr()), "marl_gru_seq_fwd")
            ctx.seq = True
            if need:
                ctx.save_for_backward(x, h0, w_ih, w_hh, out, saves, packed)
            return out
        ctx.seq = False
        gh = torch.empty(R, 3 * E, dtype=x.dtype, device=x.device)
        w_hh_t = w_hh.t()
        h = h0.contiguous()
        L, P, st = _L(), _lib.ptr, _lib.stream_ptr()
        for t in range(T):
            if tc:
                _gemm_tc(h, None, w_hh, b_hh, None, False, out=gh)
            else:
                torch.addmm(b_hh, h, w_hh_t, out=gh)
            sv = [saves[k, t].data_ptr() for k in range(4)] if need else [None] * 4
            _lib.check(L.marl_gru_cell_fwd(R, E, gi_all[t].data_ptr(), P(gh), h.data_ptr(), out[t].data_ptr(), *sv, st),
                       "marl_gru_cell_fwd")
            h = out[t]
        if need:
            ctx.save_for_backward(x, h0, w_ih, w_hh, out, saves)
        return out

    @staticmethod
    def backward(ctx, d_out):
        if ctx.seq:
            x, h0, w_ih, w_hh, out, saves, packed = ctx.saved_tensors
            T, R, E = x.shape
            d_out = d_out.contiguous()
            dgi = torch.empty(T, R, 3 * E, dtype=x.dtype, device=x.device)
            dgh = torch.empty(T, R, 3 * E, dtype=x.dtype, device=x.device)
            dh0 = torch.empty(R, E, dtype=x.dtype, device=x.device)
            h0c = h0.contiguous()
            CALLS["gru_seq_bwd"] += 1
            _lib.check(_L().marl_gru_seq_bwd(T, R, E, d_out.data_ptr(), saves.data_ptr(), out.data_ptr(), h0c.data_ptr(),
                                             packed.data_ptr(), dgi.data_ptr(), dgh.data_ptr(), dh0.data_ptr(), _lib.stream_ptr()),
                       "marl_gru_seq_bwd")
            dgi2, dgh2 = dgi.view(T * R, 3 * E), dgh.view(T * R, 3 * E)
            h_prev_all = torch.cat([h0c.unsqueeze(0), out[:-1]], dim=0).view(T * R, E)
            dx = (_gemm_tc(dgi2, None, w_ih, None, None, False, transposed=True) if _tc_t_ok(dgi2, w_ih) else torch.mm(dgi2, w_ih)).view(T, R, E)
            db_ih = torch.empty(3 * E, dtype=x.dtype, device=x.device)
            db_hh = torch.empty(3 * E, dtype=x.dtype, device=x.device)
            return (dx, dh0, wgrad(dgi2, x.view(T * R, E), dbias=db_ih), wgrad(dgh2, h_prev_all, dbias=db_hh), db_ih, db_hh)
        x, h0, w_ih, w_hh, out, saves = ctx.saved_tensors
        T, R, E = x.shape
        d_out = d_out.contiguous()
        dgi = torch.empty(T, R, 3 * E, dtype=x.dtype, device=x.device)
        dgh = torch.empty(T, R, 3 * E, dtype=x.dtype, device=x.device)
        dh = torch.zeros(R, E, dtype=x.dtype, device=x.device)
        dh_tot = torch.empty_like(dh)
        dh_prev = torch.empty_like(dh)
        h0c = h0.contiguous()
        L, st = _L(), _lib.stream_ptr()
        w_hh_T = w_hh.t().contiguous()                      # [E,3E]: "weight" of the dh_{t-1} += dgh_t @ W_hh projection
        tc = _tc_ok(dgh[0], w_hh_T, None)
        for t in range(T - 1, -1, -1):
            torch.add(d_out[t], dh, out=dh_tot)
            hp = out[t - 1] if t > 0 else h0c
            _lib.check(L.marl_gru_cell_bwd(R, E, dh_tot.data_ptr(), saves[0, t].data_ptr(), saves[1, t].data_ptr(),
                                           saves[2, t].data_ptr(), saves[3, t].data_ptr(), hp.data_ptr(),
                                           dgi[t].data_ptr(), dgh[t].data_ptr(), dh_prev.data_ptr(), st),
                       "marl_gru_cell_bwd")
            if tc:                                            # dh_{t-1} = dh_t*z + dgh_t @ W_hh
                _gemm_tc(dgh[t], None, w_hh_T, None, dh_prev, False, out=dh)
            else:
                torch.addmm(dh_prev, dgh[t], w_hh, out=dh)
        dgi2, dgh2 = dgi.view(T * R, 3 * E), dgh.view(T * R, 3 * E)
        h_prev_all = torch.cat([h0c.unsqueeze(0), out[:-1]], dim=0).view(T * R, E)
        w_ih_T = w_ih.t().contiguous()
        dx = (_gemm_tc(dgi2, None, w_ih_T, None, None, False) if _tc_ok(dgi2, w_ih_T, None) else torch.mm(dgi2, w_ih)).view(T, R, E)
        return dx, dh.clone(), torch.mm(dgi2.t(), x.view(T * R, E)), torch.mm(dgh2.t(), h_prev_all), dgi2.sum(0), dgh2.sum(0)


def gru_forward(x, h0, weights, num_layers):
    """weights: list per layer of (w_ih, w_hh, b_ih, b_hh); x [T,R,E]; h0 [L,R,E] -> (out [T,R,E], hT [L,R,E])."""
    hs = []
    for layer in range(num_layers):
        x = _GRULayer.apply(x, h0[layer], *weights[layer])
        hs.append(x[-1])
    return x, torch.stack(hs)


def spectral_sigma(W, u):
    """One power iteration of torch.nn.utils.spectral_norm (exact for the [1,E] critic head).  Returns
    (sigma, u_new, v_new); sigma is to be treated as u^T W v with u, v constants."""
    with torch.no_grad():
        v = torch.nn.functional.normalize(torch.mv(W.t(), u), dim=0, eps=1e-12)
        u2 = torch.nn.functional.normalize(torch.mv(W, v), dim=0, eps=1e-12)
        sigma = torch.dot(u2, torch.mv(W, v))
    return sigma, u2, v


class _PPOHead(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat_a, feat_c, Wa, ba, Wc_orig, bc, u, action, old_logp, adv, v_old, v_target, active, eps, ent_coef):
        R, E = feat_a.shape
        A = Wa.shape[0]
        sigma, u2, v = spectral_sigma(Wc_orig, u)
        w_eff = (Wc_orig / sigma).reshape(E).contiguous()
        dev = feat_a.device
        f32 = dict(dtype=torch.float32, device=dev)
        logp, ent, val = torch.empty(R, **f32), torch.empty(R, **f32), torch.empty(R, **f32)
        dlogits, dvalue, sums = torch.empty(R, A, **f32), torch.empty(R, **f32), torch.zeros(3, **f32)
        args = [None if t is None else t.contiguous()      # v_old None: the unclipped value loss (use_value_clip = False)
                for t in (feat_a, feat_c, Wa, ba, w_eff, bc, action, old_logp, adv, v_old, v_target, active)]
        part = torch.empty(int(_L().marl_ppo_head_workspace_bytes(R)), dtype=torch.uint8, device=dev)   # fixed-order loss sums
        _lib.check(_L().marl_ppo_head_det(R, E, A, *[_lib.ptr(t) for t in args], ctypes.c_float(eps), ctypes.c_float(ent_coef),
                                          _lib.ptr(logp), _lib.ptr(ent), _lib.ptr(val), _lib.ptr(dlogits), _lib.ptr(dvalue),
                                          _lib.ptr(sums), _lib.ptr(part), _lib.stream_ptr()), "marl_ppo_head_det")
        ctx.save_for_backward(args[0], args[1], args[2], w_eff, dlogits, dvalue, sums, sigma, u2, v)
        ctx.mark_non_differentiable(logp, ent, val, u2, v)
        return sums[0] / sums[2], sums[1] / sums[2], logp, ent, val, u2, v

    @staticmethod
    def backward(ctx, g_actor, g_critic, *_unused):
        feat_a, feat_c, Wa, w_eff, dlogits, dvalue, sums, sigma, u2, v = ctx.saved_tensors
        dl = dlogits * (g_actor / sums[2])
        dv = dvalue * (g_critic / sums[2])
        d_feat_a = torch.mm(dl, Wa)
        dWa = skinny_outer(feat_a, dl).t()               # [A, E] = dl^T feat_a in one pass over feat_a (a 1 ms SIMT sgemm otherwise)
        dba = dl.sum(0)
        d_feat_c = dv.unsqueeze(1) * w_eff.unsqueeze(0)
        dw_eff = torch.mv(feat_c.t(), dv)
        dbc = dv.sum().reshape(1)
        # W_eff = W / sigma, sigma = u^T W v  =>  dW = (dW_eff - <dW_eff, W_eff> u v^T) / sigma
        dWc = (dw_eff.unsqueeze(0) - (dw_eff * w_eff).sum() * (u2.unsqueeze(1) * v.unsqueeze(0))) / sigma
        return (d_feat_a, d_feat_c, dWa, dba, dWc, dbc) + (None,) * 9


def ppo_head(feat_a, feat_c, Wa, ba, Wc_orig, bc, u, action, old_logp, adv, v_old, v_target, active, eps, ent_coef):
    """-> (actor_loss, critic_loss, logp [R], entropy [R], value [R], u_new, v_new).  v_old = None: no value clip."""
    return _PPOHead.apply(feat_a, feat_c, Wa, ba, Wc_orig, bc, u, action, old_logp, adv, v_old, v_target, active,
                          float(eps), float(ent_coef))


def act_head(feat_a, feat_c, Wa, ba, w_eff, bc, seed, t, deterministic):
    """Rollout heads: -> (action i32 [R], action f32 [R], logp [R], value [R] or None)."""
    R, E = feat_a.shape
    dev = feat_a.device
    action = torch.empty(R, dtype=torch.int32, device=dev)
    action_f = torch.empty(R, dtype=torch.float32, device=dev)
    logp = torch.empty(R, dtype=torch.float32, device=dev)
    value = torch.empty(R, dtype=torch.float32, device=dev) if feat_c is not None else None
    _lib.check(_L().marl_act_head(R, E, Wa.shape[0], _lib.ptr(feat_a.contiguous()),
                                  _lib.ptr(feat_c.contiguous()) if feat_c is not None else None, _lib.ptr(Wa.contiguous()),
                                  _lib.ptr(ba.contiguous()), _lib.ptr(w_eff) if w_eff is not None else None,
                                  _lib.ptr(bc) if bc is not None else None, ctypes.c_uint64(seed), int(t),
                                  1 if deterministic else 0, _lib.ptr(action), _lib.ptr(action_f), _lib.ptr(logp),
                                  _lib.ptr(value), _lib.stream_ptr()), "marl_act_head")
    return action, action_f, logp, value


def clip_grad_norm_(flat_grad, max_norm):
    """In-place global-norm clip of a flat fp32 gradient arena; returns the pre-clip norm (0-dim tensor)."""
    n = flat_grad.numel()
    ws = torch.empty(int(_L().marl_clip_workspace_bytes(n)), dtype=torch.uint8, device=flat_grad.device)
    total = torch.empty(1, dtype=torch.float32, device=flat_grad.device)
    _lib.check(_L().marl_clip_grad_norm(n, _lib.ptr(flat_grad), ctypes.c_float(max_norm), _lib.ptr(ws), _lib.ptr(total),
                                        _lib.stream_ptr()), "marl_clip_grad_norm")
    return total[0]


def adam_step_(flat_param, flat_grad, exp_avg, exp_avg_sq, lr, step, betas=(0.9, 0.999), eps=1e-5):
    _lib.check(_L().marl_adam_step(flat_param.numel(), _lib.ptr(flat_param), _lib.ptr(flat_grad), _lib.ptr(exp_avg),
                                   _lib.ptr(exp_avg_sq), ctypes.c_float(lr), ctypes.c_float(betas[0]),
                                   ctypes.c_float(betas[1]), ctypes.c_float(eps), int(step), _lib.stream_ptr()),
               "marl_adam_step")
