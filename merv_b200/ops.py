"""Functional layer: torch tensors in, torch tensors out, every op one call into libmerv_fusion.so.

PyTorch is plumbing here (device memory from its caching allocator, the current CUDA stream); all arithmetic
happens in the hand-written sm_100a kernels.  CPU tensors are rejected: there is no fallback.
"""

from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ACT_GELU_ERF, ACT_NONE, MERV_BF16, MERV_F32, ROWDOT_BLOCK, PoolDesc, check, i32_array, i64_array, ptr_array

_DTYPES = {torch.float32: MERV_F32, torch.bfloat16: MERV_BF16}


def dtype_code(dtype: torch.dtype) -> int:
    try:
        return _DTYPES[dtype]
    except KeyError:
        raise TypeError(f"merv_b200 supports float32 and bfloat16 tensors, got {dtype}") from None


def _require_cuda(*tensors: torch.Tensor) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError(
                "merv_b200 runs only on CUDA (sm_100a) tensors; got a tensor on "
                f"{t.device}. There is deliberately no CPU fallback."
            )
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"tensors on different devices: {dev} vs {t.device}")
    return dev


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _rows_in_place(x: torch.Tensor) -> torch.Tensor:
    """x [B, T, K] as the kernels read or write it in place — channels contiguous, row and batch strides whole 16-byte vectors that keep
    rows and videos apart, 16-byte aligned base (e.g. the prefix slot ``buf[:, bos:bos + T]`` of the multimodal embedding buffer or its
    gradient) — or else a contiguous copy."""
    vec = 8 if x.dtype == torch.bfloat16 else 4
    B, T, K = x.shape
    if (x.stride(2) != 1 or x.stride(1) % vec or x.stride(0) % vec or x.data_ptr() % 16
            or (T > 1 and x.stride(1) < K) or (B > 1 and x.stride(0) < T * x.stride(1))):
        x = x.contiguous()
    return x


# ---- launch accounting ----------------------------------------------------------------------------------------
# kernels launched by one call of each entry point (used for bench.py's `gpu_launches` and per-kernel timing)
KERNELS_PER_CALL = {
    "merv_pool3d": 1, "merv_linear_bias_act": 1, "merv_gemm_ex": 1, "merv_fusion_query_vec": 3, "merv_affine_score_vec": 3,
    "merv_scores_from_tokens": 2, "merv_scores_from_partials": 1, "merv_softmax_weights": 1,
    "merv_softmax_mix": 1, "merv_fused_linear_mix": 1, "merv_fused_forward": 3, "merv_softmax_weights_ex": 1,
    "merv_transpose": 1, "merv_colsum": 2, "merv_mix_backward": 10, "merv_gelu": 1,
    "merv_cross_attention": 1, "merv_cross_attention_backward": 1, "merv_add_rows": 1, "merv_video_colsum": 1, "merv_pair_dot": 1, "merv_transpose_rowscale": 1, "merv_fused_backward": 10, "merv_wgrad_video": 3,
    "merv_scores_from_tokens_ex": 2, "merv_score_consts": 1, "merv_layernorm": 1, "merv_layernorm_backward": 1, "merv_concat_linear": 1,
    "merv_mix_backward_ex": 10,  # as merv_mix_backward; one more with single-token encoders, one fewer with averagetoken=False
    "merv_scalar_mix_backward": 2, "merv_scalar_fused_backward": 2,
    "merv_cross_attention_backward_ex": 1,
}


class KernelTimer:
    """Optional per-entry-point accounting: counts kernel launches and, if `timing`, brackets every library call
    with CUDA events on the launching stream (bench.py uses it for the roofline of the dominant kernel)."""

    def __init__(self, timing: bool = False) -> None:
        self.timing = timing
        self.launches = 0
        self.calls = {}
        self._events = []

    def __enter__(self):
        global _timer
        self._prev, _timer = _timer, self
        return self

    def __exit__(self, *exc):
        global _timer
        _timer = self._prev
        return False

    def durations_ms(self):
        """{entry point: [ms per call]} — synchronises."""
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1 in self._events:
            out.setdefault(name, []).append(e0.elapsed_time(e1))
        return out


_timer: Optional[KernelTimer] = None


def _call(name, fn, *args) -> None:
    t = _timer
    if t is None:
        check(fn(*args))
        return
    t.launches += KERNELS_PER_CALL[name]
    t.calls[name] = t.calls.get(name, 0) + 1
    if t.timing:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(fn(*args))
        e1.record()
        t._events.append((name, e0, e1))
    else:
        check(fn(*args))


# ------------------------------------------------------------------------------------------------------------
def pool3d(
    xs: Sequence[torch.Tensor], out_frames: Sequence[int], out_size: int,
    score_vecs: Optional[Sequence[torch.Tensor]] = None, max_ctas: int = 0, batch_index: Optional[torch.Tensor] = None,
    shifts: Optional[Sequence[Tuple[int, int, int]]] = None, outs: Optional[Sequence[torch.Tensor]] = None,
) -> Tuple[List[torch.Tensor], Optional[List[torch.Tensor]]]:
    """Adaptive 3-D average pooling of every encoder's [B, F, N, C] features in ONE launch -> [B, T*S*S, C].

    Reference: AveragePooling3DProjector.forward, merv/util/nn_utils.py:320-329.  With `score_vecs` (fp32 [C_e] each)
    also returns per-encoder partial dot products [B, parts_e] of the pooled tokens with that vector.  `batch_index`
    (int32 [B']) selects/reorders the videos read from every x (the `multimodal_indices` gather of merv.py:572, fused).
    `shifts` ((frames, rows, columns) per entry): the windows read x displaced by that much, out-of-grid positions counting as zero
    (one tap of a zero-padded convolution, see `pool3d_conv_taps`).  `outs`: [B, T*S*S, C] destinations (any row / batch stride,
    channels contiguous) instead of fresh tensors.
    """
    lib = _lib.load()
    dev = _require_cuda(*xs, *(score_vecs or []), batch_index)
    src_B = xs[0].shape[0]
    if batch_index is not None:
        assert batch_index.dtype == torch.int32 and batch_index.dim() == 1 and batch_index.is_contiguous()
    B = src_B if batch_index is None else batch_index.numel()
    code = dtype_code(xs[0].dtype)
    n = len(xs)
    descs = (PoolDesc * n)()
    ys, keep = [], []
    with torch.cuda.device(dev):
        for i, (x, T) in enumerate(zip(xs, out_frames)):
            assert x.dim() == 4, f"expected [B, F, N, C] features, got {tuple(x.shape)}"
            assert x.shape[0] == src_B and x.dtype == xs[0].dtype
            if x.stride(3) != 1 or any(s % 8 for s in x.stride()[:3]):
                x = x.contiguous()
            keep.append(x)
            _, F, N, Cc = x.shape
            H = int(math.sqrt(N))  # nn_utils.py:322
            assert H * H == N, f"patch count {N} is not a perfect square (einops would reject it at nn_utils.py:323-327)"
            if outs is not None:
                y = outs[i]
                assert y.shape == (B, T * out_size * out_size, Cc) and y.dtype == x.dtype and y.stride(2) == 1 and y.device == x.device
            else:
                y = torch.empty((B, T * out_size * out_size, Cc), dtype=x.dtype, device=dev)
            d = descs[i]
            if shifts is not None:
                d.shift_f, d.shift_h, d.shift_w = (int(v) for v in shifts[i])
            d.x, d.y, d.score_vec, d.score_partial = x.data_ptr(), y.data_ptr(), None, None
            d.batch_index, d.src_batch = _p(batch_index), src_B
            d.F, d.H, d.W, d.C, d.T, d.S = F, H, H, Cc, T, out_size
            d.x_batch_stride, d.x_frame_stride, d.x_token_stride = x.stride(0), x.stride(1), x.stride(2)
            d.y_batch_stride, d.y_row_stride = y.stride(0), y.stride(1)
            ys.append(y)
        partials = None
        if score_vecs is not None:
            parts = i32_array([0] * n)
            check(lib.merv_pool3d_score_parts(descs, n, code, parts))
            partials = []
            for i, sv in enumerate(score_vecs):
                assert sv.dtype == torch.float32 and sv.numel() == xs[i].shape[3] and sv.is_contiguous()
                pt = torch.empty((B, parts[i]), dtype=torch.float32, device=dev)
                descs[i].score_vec, descs[i].score_partial = sv.data_ptr(), pt.data_ptr()
                partials.append(pt)
        _call('merv_pool3d', lib.merv_pool3d, descs, n, B, code, max_ctas, _stream())
    return ys, partials


CONV_TAPS = [(df, dh, dw) for df in (-1, 0, 1) for dh in (-1, 0, 1) for dw in (-1, 0, 1)]  # Conv3d kernel index (kf, kh, kw) = shift + 1


def pool3d_conv_taps(x: torch.Tensor, out_frames: int, out_size: int) -> torch.Tensor:
    """A [B, T*S*S, 27*C]: the adaptive average pooling of the 27 displaced copies of x [B, F, N, C] (zero outside the grid), tap-major
    columns — the operand that turns `AdaptiveAvgPool3d(Conv3d(C, K, kernel_size=3, padding=1)(x))` (Convolutional3DProjector,
    merv/util/nn_utils.py:349-352,364) into ONE GEMM on the pooled grid: pooling is linear, so it commutes with the convolution's sum
    over taps, and pooling first cuts the contraction from F*H*W to T*S*S positions per video (4x fewer at merv-full shapes)."""
    B, _, _, Cc = x.shape
    n_tok = out_frames * out_size * out_size
    A = torch.empty((B, n_tok, len(CONV_TAPS) * Cc), dtype=x.dtype, device=x.device)
    per = _lib.MAX_ENCODERS
    for t0 in range(0, len(CONV_TAPS), per):
        taps = CONV_TAPS[t0:t0 + per]
        pool3d([x] * len(taps), [out_frames] * len(taps), out_size, shifts=taps,
               outs=[A[:, :, (t0 + i) * Cc:(t0 + i + 1) * Cc] for i in range(len(taps))])
    return A


def linear_bias_act(
    a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], act: int = ACT_NONE,
    rowdot_vec: Optional[torch.Tensor] = None,
) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """y = act(a @ w.T + bias) for a [..., K], w [N, K]; optional row-dot partials [M, ceil(N/128)] (bf16 path).

    Reference: nn.Linear (+ nn.GELU) in merv/util/nn_utils.py:31-32,46-55,97-108.
    """
    lib = _lib.load()
    dev = _require_cuda(a, w, bias, rowdot_vec)
    code = dtype_code(a.dtype)
    assert w.dtype == a.dtype and (bias is None or bias.dtype == a.dtype), "weights must be in the activation dtype"
    K = a.shape[-1]
    N = w.shape[0]
    assert w.shape[1] == K, f"weight {tuple(w.shape)} does not match input features {K}"
    a2 = a.reshape(-1, K)
    if a2.stride(1) != 1:
        a2 = a2.contiguous()
    if w.stride(1) != 1:
        w = w.contiguous()
    M = a2.shape[0]
    with torch.cuda.device(dev):
        y = torch.empty((M, N), dtype=a.dtype, device=dev)
        rd = None
        if rowdot_vec is not None:
            assert rowdot_vec.dtype == torch.float32 and rowdot_vec.numel() == N
            rd = torch.empty((M, (N + ROWDOT_BLOCK - 1) // ROWDOT_BLOCK), dtype=torch.float32, device=dev)
        _call('merv_linear_bias_act', lib.merv_linear_bias_act, a2.data_ptr(), a2.stride(0), w.data_ptr(), w.stride(0), _p(bias), y.data_ptr(), y.stride(0),
                                       M, N, K, act, code, _p(rowdot_vec), _p(rd), _stream())
    return y.reshape(*a.shape[:-1], N), rd


def gemm_ex(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, act: int = ACT_NONE, a_t: bool = False,
            w_t: bool = False) -> torch.Tensor:
    """y [M, N] = act(A W^T + bias) on the tcgen05 GEMM (bf16) with either operand handed over TRANSPOSED, without a copy:
    ``a_t``: ``a`` is A^T, a [K, M] matrix; ``w_t``: ``w`` is W^T, a [K, N] matrix (row-major, any 16-byte aligned row stride).

    The backward of a Linear (autograd of nn_utils.py:31-32,46-55): ``dW = gemm_ex(dY, X, a_t=True, w_t=True)`` (contraction over the
    tokens) and ``dX = gemm_ex(dY, W, w_t=True)`` — no transposed copies of dY, X or W."""
    lib = _lib.load()
    dev = _require_cuda(a, w, bias)
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and (bias is None or bias.dtype == torch.bfloat16), "gemm_ex is bf16 only"
    assert a.dim() == 2 and w.dim() == 2
    a = a if a.stride(1) == 1 and a.stride(0) % 8 == 0 and a.data_ptr() % 16 == 0 else a.contiguous()
    w = w if w.stride(1) == 1 and w.stride(0) % 8 == 0 and w.data_ptr() % 16 == 0 else w.contiguous()
    K, M = (a.shape if a_t else a.shape[::-1])
    Kw, N = (w.shape if w_t else w.shape[::-1])
    assert K == Kw, f"contraction lengths differ: {K} vs {Kw}"
    with torch.cuda.device(dev):
        y = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
        _call('merv_gemm_ex', lib.merv_gemm_ex, a.data_ptr(), a.stride(0), int(a_t), w.data_ptr(), w.stride(0), int(w_t), _p(bias), y.data_ptr(),
              y.stride(0), M, N, K, act, _stream())
    return y


def fusion_query_vec(Q: torch.Tensor, Wq: torch.Tensor, Wk: torch.Tensor, in_proj_bias: Optional[torch.Tensor]) -> torch.Tensor:
    """u = Wk^T (Wq Q^T + b_q) / sqrt(embed), fp32 [llm_dim] (SURVEY.md §3.3; nn_utils.py:499-512)."""
    lib = _lib.load()
    dev = _require_cuda(Q, Wq, Wk, in_proj_bias)
    code = dtype_code(Q.dtype)
    embed, llm_dim = Wk.shape
    assert Wq.shape == (embed, embed) and Q.numel() == embed
    Q, Wq, Wk = Q.contiguous(), Wq.contiguous(), Wk.contiguous()
    with torch.cuda.device(dev):
        u = torch.empty(llm_dim, dtype=torch.float32, device=dev)
        n = -(-embed // 4) * 4 + lib.merv_gemv_t_workspace(embed, llm_dim)
        ws = torch.empty(n, dtype=torch.float32, device=dev)
        _call('merv_fusion_query_vec', lib.merv_fusion_query_vec, Q.data_ptr(), Wq.data_ptr(), Wk.data_ptr(), _p(in_proj_bias), u.data_ptr(), ws.data_ptr(),
                                        n, embed, llm_dim, code, _stream())
    return u


def affine_score_vec(W: torch.Tensor, bias: Optional[torch.Tensor], u: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(v, c) with u . (W x + b) == v . x + c: v = W^T u [K] fp32, c = u . b [1] fp32."""
    lib = _lib.load()
    dev = _require_cuda(W, bias, u)
    N, K = W.shape
    if W.stride(1) != 1:
        W = W.contiguous()
    with torch.cuda.device(dev):
        v = torch.empty(K, dtype=torch.float32, device=dev)
        c = torch.empty(1, dtype=torch.float32, device=dev)
        n = lib.merv_gemv_t_workspace(N, K)
        ws = torch.empty(n, dtype=torch.float32, device=dev) if n else None
        _call('merv_affine_score_vec', lib.merv_affine_score_vec, W.data_ptr(), W.stride(0), _p(bias), u.data_ptr(), v.data_ptr(), c.data_ptr(), _p(ws), n,
                                        N, K, dtype_code(W.dtype), _stream())
    return v, c


def scores_from_tokens(Vs: Sequence[torch.Tensor], u: torch.Tensor, token_length: int, per_token_u: bool = False,
                       consts: Optional[torch.Tensor] = None, mean: bool = True) -> torch.Tensor:
    """scores[b, e] = mean_t(u . V_e[b, t, :]) (+ consts[e]) read from the tokens (general path).

    ``per_token_u``: u is [T*K] with one row per token and nothing is averaged unless ``mean`` — the averagetoken=False
    branch (nn_utils.py:514-518).  ``consts`` (fp32 [E]): additive constants, u . pe[e] for positional_embedding=True
    (nn_utils.py:510-511)."""
    lib = _lib.load()
    dev = _require_cuda(*Vs, u, consts)
    B, _, K = Vs[0].shape
    E = len(Vs)
    Vs = [v.contiguous() for v in Vs]
    assert u.dtype == torch.float32 and u.is_contiguous() and u.numel() == (token_length * K if per_token_u else K)
    assert consts is None or (consts.dtype == torch.float32 and consts.is_contiguous() and consts.numel() == E)
    with torch.cuda.device(dev):
        scores = torch.empty((B, E), dtype=torch.float32, device=dev)
        n = lib.merv_scores_from_tokens_workspace(B, E, token_length, K)
        ws = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
        if not per_token_u and consts is None and mean:
            _call('merv_scores_from_tokens', lib.merv_scores_from_tokens, ptr_array([v.data_ptr() for v in Vs]), i32_array([v.shape[1] for v in Vs]),
                  u.data_ptr(), scores.data_ptr(), ws.data_ptr(), n, B, E, token_length, K, dtype_code(Vs[0].dtype), _stream())
        else:
            _call('merv_scores_from_tokens_ex', lib.merv_scores_from_tokens_ex, ptr_array([v.data_ptr() for v in Vs]),
                  i32_array([v.shape[1] for v in Vs]), u.data_ptr(), K if per_token_u else 0, _p(consts), int(mean), scores.data_ptr(),
                  ws.data_ptr(), n, B, E, token_length, K, dtype_code(Vs[0].dtype), _stream())
    return scores


def score_consts(pe: torch.Tensor, u: torch.Tensor, c_in: Optional[Sequence[Optional[torch.Tensor]]] = None) -> torch.Tensor:
    """c[e] = u . pe[e] (+ c_in[e]) — what positional_embedding=True adds to encoder e's score (nn_utils.py:510-511)."""
    lib = _lib.load()
    dev = _require_cuda(pe, u, *(c_in or []))
    E, K = pe.shape
    if pe.stride(1) != 1:
        pe = pe.contiguous()
    assert u.dtype == torch.float32 and u.numel() == K and u.is_contiguous()
    with torch.cuda.device(dev):
        c = torch.empty(E, dtype=torch.float32, device=dev)
        cptr = ptr_array([_p(t) for t in c_in]) if c_in is not None else None
        _call('merv_score_consts', lib.merv_score_consts, pe.data_ptr(), pe.stride(0), u.data_ptr(), cptr, c.data_ptr(), E, K, dtype_code(pe.dtype),
              _stream())
    return c


def _segments(xs: Sequence[torch.Tensor]):
    lead = xs[0].shape[:-1]
    xs = [x.reshape(-1, x.shape[-1]) for x in xs]
    vec = 8 if xs[0].dtype == torch.bfloat16 else 4
    xs = [x if x.stride(1) == 1 and x.stride(0) % vec == 0 and x.data_ptr() % 16 == 0 else x.contiguous() for x in xs]
    M = xs[0].shape[0]
    assert all(x.shape[0] == M and x.dtype == xs[0].dtype for x in xs), "segments must share rows and dtype"
    return lead, xs, M


def layernorm(xs: Sequence[torch.Tensor], weight: Optional[torch.Tensor], bias: Optional[torch.Tensor], eps: float = 1e-5) -> torch.Tensor:
    """LayerNorm over the last dimension of concat(xs, -1) without building the concatenation: [..., sum K_s].

    nn.LayerNorm in front of a projector (pre_proj_layernorm, nn_utils.py:26-29) with one segment; the LayerNorm(E * llm_dim)
    of feature_fusion == "concat_channel_ln" (merv.py:219-223,603-606) with E segments."""
    lib = _lib.load()
    dev = _require_cuda(*xs, weight, bias)
    lead, xs, M = _segments(xs)
    total = sum(x.shape[1] for x in xs)
    dt = xs[0].dtype
    assert weight is None or (weight.dtype == dt and weight.numel() == total and weight.is_contiguous())
    assert bias is None or (bias.dtype == dt and bias.numel() == total and bias.is_contiguous())
    with torch.cuda.device(dev):
        y = torch.empty((M, total), dtype=dt, device=dev)
        _call('merv_layernorm', lib.merv_layernorm, ptr_array([x.data_ptr() for x in xs]), i64_array([x.stride(0) for x in xs]),
              i32_array([x.shape[1] for x in xs]), len(xs), _p(weight), _p(bias), float(eps), y.data_ptr(), y.stride(0), M, dtype_code(dt), _stream())
    return y.view(*lead, total)


def layernorm_backward(xs: Sequence[torch.Tensor], dy: torch.Tensor, weight: Optional[torch.Tensor], eps: float = 1e-5,
                       need_dx: bool = True, need_params: bool = True):
    """Backward of `layernorm`: returns (dx [M, sum K_s] | None, dweight | None, dbias | None) in the compute dtype."""
    lib = _lib.load()
    dev = _require_cuda(*xs, dy, weight)
    _, xs, M = _segments(xs)
    total = sum(x.shape[1] for x in xs)
    dt = xs[0].dtype
    dy = dy.reshape(M, total)
    if dy.dtype != dt:
        dy = dy.to(dt)
    if dy.stride(1) != 1 or dy.stride(0) % (8 if dt == torch.bfloat16 else 4) or dy.data_ptr() % 16:
        dy = dy.contiguous()
    with torch.cuda.device(dev):
        dx = torch.empty((M, total), dtype=dt, device=dev) if need_dx else None
        gx = torch.empty((M, total), dtype=dt, device=dev) if need_params else None
        _call('merv_layernorm_backward', lib.merv_layernorm_backward, ptr_array([x.data_ptr() for x in xs]), i64_array([x.stride(0) for x in xs]),
              i32_array([x.shape[1] for x in xs]), len(xs), dy.data_ptr(), dy.stride(0), _p(weight), float(eps), _p(dx),
              dx.stride(0) if need_dx else 0, _p(gx), gx.stride(0) if need_params else 0, M, dtype_code(dt), _stream())
    if not need_params:
        return dx, None, None
    return dx, colsum(gx), colsum(dy)


def scores_from_partials(partials: Sequence[torch.Tensor], consts: Optional[Sequence[Optional[torch.Tensor]]], B: int, T: int) -> torch.Tensor:
    """scores[b,e] = (1/T) * sum(partials_e[b]) + c_e from the pool kernel's / GEMM epilogue's partial dot products."""
    lib = _lib.load()
    dev = _require_cuda(*partials)
    E = len(partials)
    counts = [p.numel() // B for p in partials]
    with torch.cuda.device(dev):
        scores = torch.empty((B, E), dtype=torch.float32, device=dev)
        cptr = ptr_array([_p(c) for c in consts]) if consts is not None else None
        _call('merv_scores_from_partials', lib.merv_scores_from_partials, ptr_array([p.data_ptr() for p in partials]), i32_array(counts),
              cptr, scores.data_ptr(), B, E, T, _stream())
    return scores


def num_sms() -> int:
    return _lib.load().merv_num_sms()


def softmax_weights(
    scores: torch.Tensor, biases: Optional[Sequence[Optional[torch.Tensor]]] = None, N: int = 0,
    out: Optional[torch.Tensor] = None,
) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """weights = softmax(scores, -1) (fp32) and, if `biases` is given, bias_mix[b] = sum_e weights[b,e] * bias_e (fp32 [B, N])."""
    lib = _lib.load()
    dev = _require_cuda(scores)
    B, E = scores.shape
    with torch.cuda.device(dev):
        weights = out if out is not None else torch.empty((B, E), dtype=torch.float32, device=dev)
        assert weights.shape == (B, E) and weights.dtype == torch.float32 and weights.is_contiguous()
        bias_mix, bptr, code = None, None, MERV_F32
        if biases is not None:
            bias_mix = torch.empty((B, N), dtype=torch.float32, device=dev)
            bptr = ptr_array([_p(b) for b in biases])
            present = [b for b in biases if b is not None]
            code = dtype_code(present[0].dtype) if present else MERV_F32
        _call('merv_softmax_weights', lib.merv_softmax_weights, scores.data_ptr(), weights.data_ptr(), bptr, _p(bias_mix), B, E, N, code, _stream())
    return weights, bias_mix


def softmax_mix(
    Vs: Sequence[torch.Tensor], token_length: int, scores: Optional[torch.Tensor] = None, weights: Optional[torch.Tensor] = None,
    out: Optional[torch.Tensor] = None,
) -> Tuple[torch.Tensor, torch.Tensor]:
    """out[b,t,:] = sum_e w[b,e] V_e[b,t,:] with w = softmax(scores) computed in-kernel (or given `weights`).

    Reference: torch.stack + torch.bmm at merv/util/nn_utils.py:503,521.  Returns (out [B,T,K], weights fp32 [B,E]).
    `out`: optional [B, T, K] destination (any row / batch stride), e.g. the prefix slot of the multimodal embedding buffer; written in
    place when the kernel can address it (include/merv_fusion.h: merv_softmax_mix_ex), otherwise through a contiguous copy.
    """
    lib = _lib.load()
    dev = _require_cuda(*Vs, scores, weights, out)
    assert (scores is None) != (weights is None)
    B, _, K = Vs[0].shape
    E = len(Vs)
    Vs = [v.contiguous() for v in Vs]
    with torch.cuda.device(dev):
        dst = torch.empty((B, token_length, K), dtype=Vs[0].dtype, device=dev) if out is None else _rows_in_place(out)
        assert dst.shape == (B, token_length, K) and dst.dtype == Vs[0].dtype, f"out must be {Vs[0].dtype} [{B}, {token_length}, {K}]"
        if weights is None:
            weights = torch.empty((B, E), dtype=torch.float32, device=dev)
        _call('merv_softmax_mix', lib.merv_softmax_mix_ex, ptr_array([v.data_ptr() for v in Vs]), i32_array([v.shape[1] for v in Vs]), _p(scores),
              weights.data_ptr(), dst.data_ptr(), dst.stride(1), dst.stride(0), B, E, token_length, K, dtype_code(Vs[0].dtype), _stream())
    if out is not None and dst is not out:
        out.copy_(dst)
        dst = out
    return dst, weights


def fused_linear_mix(
    As: Sequence[torch.Tensor], Ws: Sequence[torch.Tensor], scale: torch.Tensor, bias_mix: Optional[torch.Tensor],
    rows_per_video: int, out: Optional[torch.Tensor] = None, max_ctas: int = 0, peer_out_ptrs: Optional[Sequence[int]] = None,
    multicast_out_ptr: Optional[int] = None,
) -> torch.Tensor:
    """out[m] = sum_s scale[m // rows_per_video, s] * (A_s[m] @ W_s.T) + bias_mix[m // rows_per_video]  (bf16, tcgen05).

    `peer_out_ptrs`: device addresses (peer-mapped, e.g. from torch symmetric memory) of the same [M, N] block in other
    ranks' buffers; every output tile is then also stored there over NVLink (fused all-gather, see merv_b200.parallel).

    `multicast_out_ptr`: NVSwitch multicast address of the same block (torch symmetric memory's ``multicast_ptr`` + block offset);
    every output box is then written ONCE with multimem.st and the switch replicates it into every rank's buffer, `out` included.

    `out` may be a preallocated [M, N] matrix (row stride >= N) or a [B, rows_per_video, N] view with an arbitrary batch
    stride, e.g. `embeddings[:, bos:bos + T, :]` of the multimodal embedding buffer (merv.py:633-640): the prefix is then
    written in place instead of being concatenated afterwards.
    """
    lib = _lib.load()
    dev = _require_cuda(*As, *Ws, scale, bias_mix, out)
    assert all(a.dtype == torch.bfloat16 for a in As) and all(w.dtype == torch.bfloat16 for w in Ws), "fused path is bf16 only"
    As = [a.reshape(-1, a.shape[-1]) for a in As]
    As = [a if a.stride(1) == 1 else a.contiguous() for a in As]
    Ws = [w if w.stride(1) == 1 else w.contiguous() for w in Ws]
    M, N = As[0].shape[0], Ws[0].shape[0]
    assert all(a.shape[0] == M for a in As), f"every segment must have the same {M} rows, got {[a.shape[0] for a in As]}"
    assert all(w.shape[0] == N and w.shape[1] == a.shape[1] for a, w in zip(As, Ws)), "weights must be [N, K_s] for A_s [M, K_s]"
    assert scale.dtype == torch.float32 and scale.is_contiguous() and scale.shape == (M // rows_per_video, len(As))
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
        assert out.dtype == torch.bfloat16 and out.stride(-1) == 1
        if out.dim() == 3:
            assert out.shape == (M // rows_per_video, rows_per_video, N)
            ldo, batch_stride = out.stride(1), out.stride(0)
        else:
            assert out.shape == (M, N)
            ldo, batch_stride = out.stride(0), 0
        peers = list(peer_out_ptrs or [])
        if multicast_out_ptr:
            assert not peers and out.is_contiguous(), "multicast output: one contiguous block, no unicast peers"
            _call('merv_fused_linear_mix', lib.merv_fused_linear_mix_multicast, ptr_array([a.data_ptr() for a in As]), i64_array([a.stride(0) for a in As]),
                  ptr_array([w.data_ptr() for w in Ws]), i64_array([w.stride(0) for w in Ws]), i32_array([a.shape[1] for a in As]), len(As),
                  scale.data_ptr(), _p(bias_mix), out.data_ptr(), N, M, N, rows_per_video, max_ctas, multicast_out_ptr, _stream())
            return out
        _call('merv_fused_linear_mix', lib.merv_fused_linear_mix_gather, ptr_array([a.data_ptr() for a in As]), i64_array([a.stride(0) for a in As]),
              ptr_array([w.data_ptr() for w in Ws]), i64_array([w.stride(0) for w in Ws]), i32_array([a.shape[1] for a in As]), len(As),
              scale.data_ptr(), _p(bias_mix), out.data_ptr(), ldo, batch_stride, M, N, rows_per_video, max_ctas,
              ptr_array(peers) if peers else None, len(peers), _stream())
    return out


def concat_linear(Ys: Sequence[torch.Tensor], weight: torch.Tensor, bias: Optional[torch.Tensor], out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """concat(Ys, dim=-1) @ weight.T + bias without building the concatenation (one K-segmented tcgen05 GEMM, bf16).

    feature_fusion == "concat_channel": merv.py:603-606 with the LinearProjector of merv.py:217-218."""
    lib = _lib.load()
    dev = _require_cuda(*Ys, weight, bias, out)
    assert all(y.dtype == torch.bfloat16 for y in Ys) and weight.dtype == torch.bfloat16, "concat_linear is bf16 only"
    lead = Ys[0].shape[:-1]
    Ys = [y.reshape(-1, y.shape[-1]) for y in Ys]
    Ys = [y if y.stride(1) == 1 else y.contiguous() for y in Ys]
    weight = weight if weight.stride(1) == 1 else weight.contiguous()
    M, N = Ys[0].shape[0], weight.shape[0]
    assert all(y.shape[0] == M for y in Ys) and sum(y.shape[1] for y in Ys) == weight.shape[1], "concat_linear: shapes do not add up"
    with torch.cuda.device(dev):
        if out is None:
            out = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
        assert out.dtype == torch.bfloat16 and out.shape == (M, N) and out.stride(1) == 1
        _call('merv_concat_linear', lib.merv_concat_linear, ptr_array([y.data_ptr() for y in Ys]), i64_array([y.stride(0) for y in Ys]),
              weight.data_ptr(), weight.stride(0), i32_array([y.shape[1] for y in Ys]), len(Ys), _p(bias), out.data_ptr(), out.stride(0), M, N, _stream())
    return out.view(*lead, N)


class FusedLinearPlan:
    """Pre-built `merv_fused_desc` for the whole affine path (pool -> scores -> softmax -> fused GEMM) at fixed shapes:
    one FFI crossing per forward instead of ~20 Python-level operations.  Matters at small batch (generate runs the path
    once per video at B = 1), where host time per launch dominates.  Workspaces are owned by the plan and reused, so a
    plan is bound to one stream."""

    def __init__(self, xs: Sequence[torch.Tensor], out_frames: Sequence[int], out_size: int, vs: Sequence[torch.Tensor],
                 cs: Sequence[torch.Tensor], Ws: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]], B: int, src_B: int):
        lib = _lib.load()
        dev = _require_cuda(*xs, *vs, *cs, *Ws)
        E = len(xs)
        assert 1 <= E <= _lib.MAX_SEGMENTS
        self.dev, self.E, self.B, self.src_B = dev, E, B, src_B
        d = self.desc = _lib.FusedDesc()
        N = Ws[0].shape[0]
        T_tok = out_frames[0] * out_size * out_size
        d.num_encoders, d.B, d.N, d.rows_per_video = E, B, N, T_tok
        self.keep = [vs, cs, Ws, biases]  # the descriptor holds raw pointers into these
        with torch.cuda.device(dev):
            self.pooled, self.partials = [], []
            for e, (x, T) in enumerate(zip(xs, out_frames)):
                _, F, Np, Cc = x.shape
                H = int(math.sqrt(Np))
                assert H * H == Np, f"patch count {Np} is not a perfect square"
                y = torch.empty((B, T * out_size * out_size, Cc), dtype=torch.bfloat16, device=dev)
                pd = d.pool[e]
                pd.y, pd.score_vec = y.data_ptr(), vs[e].data_ptr()
                pd.F, pd.H, pd.W, pd.C, pd.T, pd.S = F, H, H, Cc, T, out_size
                pd.x_batch_stride, pd.x_frame_stride, pd.x_token_stride = x.stride(0), x.stride(1), x.stride(2)
                pd.y_batch_stride, pd.y_row_stride = y.stride(0), y.stride(1)
                pd.src_batch = src_B
                self.pooled.append(y)
                d.W[e], d.ldw[e], d.bias[e], d.c[e] = Ws[e].data_ptr(), Ws[e].stride(0), _p(biases[e]), cs[e].data_ptr()
            parts = i32_array([0] * E)
            check(lib.merv_pool3d_score_parts(d.pool, E, MERV_BF16, parts))
            for e in range(E):
                pt = torch.empty((B, parts[e]), dtype=torch.float32, device=dev)
                d.pool[e].score_partial, d.parts[e] = pt.data_ptr(), parts[e]
                self.partials.append(pt)
            self.scores = torch.empty((B, E), dtype=torch.float32, device=dev)
            self.weights = torch.empty((B, E), dtype=torch.float32, device=dev)
            self.bias_mix = torch.empty((B, N), dtype=torch.float32, device=dev)
            d.scores, d.weights, d.bias_mix = self.scores.data_ptr(), self.weights.data_ptr(), self.bias_mix.data_ptr()
        self.N, self.T_tok = N, T_tok
        self.x_meta = [(tuple(x.shape), tuple(x.stride())) for x in xs]
        self.fn = lib.merv_fused_forward

    def rebind(self, vs: Sequence[torch.Tensor], cs: Sequence[torch.Tensor], Ws: Sequence[torch.Tensor],
               biases: Sequence[Optional[torch.Tensor]]) -> None:
        """Point the plan at a new version of the parameters (same shapes): workspaces are kept, no new plan is built."""
        d = self.desc
        assert len(Ws) == self.E and all(w.shape[0] == self.N and w.shape[1] == d.pool[e].C and w.dtype == torch.bfloat16 for e, w in enumerate(Ws))
        _require_cuda(*vs, *cs, *Ws, *biases)
        self.keep = [vs, cs, Ws, biases]
        for e in range(self.E):
            d.pool[e].score_vec = vs[e].data_ptr()
            d.W[e], d.ldw[e], d.bias[e], d.c[e] = Ws[e].data_ptr(), Ws[e].stride(0), _p(biases[e]), cs[e].data_ptr()

    def run(self, xs: Sequence[torch.Tensor], out: Optional[torch.Tensor], batch_index: Optional[torch.Tensor], xs_checked: bool = False):
        """`xs_checked`: the caller looked this plan up under the shapes, strides, dtype and device of `xs` (MervFusion's per-call
        cache key), so they need not be compared again — at B = 1 the call is host-bound and every microsecond of Python shows."""
        d = self.desc
        # the descriptor was built for these shapes / strides and this device: anything else would read or write out of bounds
        if len(xs) != self.E:
            raise ValueError(f"plan was built for {self.E} encoders, got {len(xs)}")
        for x, (shape, stride) in (() if xs_checked else zip(xs, self.x_meta)):
            if tuple(x.shape) != shape or tuple(x.stride()) != stride or x.dtype != torch.bfloat16 or x.device != self.dev:
                raise ValueError(f"plan was built for bf16 features {shape} with strides {stride} on {self.dev}, "
                                 f"got {x.dtype} {tuple(x.shape)} with strides {tuple(x.stride())} on {x.device}")
        if batch_index is not None:
            if (batch_index.dtype != torch.int32 or batch_index.dim() != 1 or not batch_index.is_contiguous() or batch_index.device != self.dev
                    or batch_index.numel() != self.B):
                raise ValueError(f"batch_index must be a contiguous int32 [{self.B}] tensor on {self.dev}, got {batch_index.dtype} "
                                 f"{tuple(batch_index.shape)} on {batch_index.device}")
        elif self.B != self.src_B:
            raise ValueError(f"plan gathers {self.B} of {self.src_B} videos: batch_index is required")
        if out is not None and (out.shape != (self.B, self.T_tok, self.N) or out.dtype != torch.bfloat16 or out.stride(2) != 1
                                or out.stride(1) % 8 or out.stride(0) % 8 or out.device != self.dev):
            raise ValueError(f"out must be a bf16 [{self.B}, {self.T_tok}, {self.N}] view with contiguous, 16-byte aligned rows on {self.dev}, "
                             f"got {out.dtype} {tuple(out.shape)} strides {tuple(out.stride())} on {out.device}")
        with torch.cuda.device(self.dev):
            if out is None:
                out = torch.empty((self.B, self.T_tok, self.N), dtype=torch.bfloat16, device=self.dev)
            w16 = torch.empty((self.B, self.E), dtype=torch.bfloat16, device=self.dev)
            bi = _p(batch_index)
            for e, x in enumerate(xs):
                d.pool[e].x, d.pool[e].batch_index = x.data_ptr(), bi
            d.out, d.ldo, d.out_batch_stride, d.weights_bf16 = out.data_ptr(), out.stride(1), out.stride(0), w16.data_ptr()
            _call('merv_fused_forward', self.fn, d, _stream())
        return out, w16


# ---- backward building blocks (SURVEY.md §8 f-1) ------------------------------------------------------------------
def transpose(x: torch.Tensor, pad: bool = False, row_scale: Optional[torch.Tensor] = None, rows_per_scale: int = 1) -> torch.Tensor:
    """[R, C] -> contiguous [C, R].  ``pad``: the result is [C, R'] with R' = R rounded up to one 16-byte vector and zeros in the
    extra columns — as the K-major operand of a GEMM whose contraction runs over R (dW = dY^T X over the token rows) it then meets
    the GEMM's K % 8 (bf16) / K % 4 (fp32) requirement whatever the number of tokens.  ``row_scale`` (fp32, one entry per
    ``rows_per_scale`` rows, any stride): y[c, r] = row_scale[r // rows_per_scale] * x[r, c] — the per-video mixing weight applied
    to the pooled tokens in the fused backward."""
    lib = _lib.load()
    dev = _require_cuda(x, row_scale)
    assert x.dim() == 2 and x.stride(1) == 1
    R, Cc = x.shape
    vec = 8 if x.dtype == torch.bfloat16 else 4
    Rp = -(-R // vec) * vec if pad else R
    with torch.cuda.device(dev):
        y = torch.empty((Cc, Rp), dtype=x.dtype, device=dev)
        if Rp == R and row_scale is None:
            _call('merv_transpose', lib.merv_transpose, x.data_ptr(), y.data_ptr(), R, Cc, x.stride(0), y.stride(0), dtype_code(x.dtype), _stream())
        else:
            if row_scale is not None:
                assert row_scale.dtype == torch.float32 and row_scale.dim() == 1 and row_scale.numel() * rows_per_scale >= R
            _call('merv_transpose_rowscale', lib.merv_transpose_rowscale, x.data_ptr(), y.data_ptr(), R, Rp, Cc, x.stride(0), y.stride(0),
                  _p(row_scale), row_scale.stride(0) if row_scale is not None else 0, rows_per_scale, dtype_code(x.dtype), _stream())
    return y


def cross_attention(q: torch.Tensor, kv: torch.Tensor, batches: int, heads: int, scale: Optional[float] = None) -> torch.Tensor:
    """Multi-head cross attention of `q` [n_q, C] (the same learned queries for every batch entry) or [batches, n_q, C] against
    kv [batches * n_kv, 2C] = [K | V] rows (CrossAttention.forward, nn_utils.py:393-412) -> [batches, n_q, C]."""
    lib = _lib.load()
    dev = _require_cuda(q, kv)
    C_ = q.shape[-1]
    assert kv.dim() == 2 and kv.shape[1] == 2 * C_ and kv.shape[0] % max(batches, 1) == 0 and C_ % heads == 0 and q.dtype == kv.dtype
    n_q, n_kv, hd = q.shape[-2], kv.shape[0] // max(batches, 1), C_ // heads
    q = q if q.stride(-1) == 1 else q.contiguous()
    kv = kv if kv.stride(1) == 1 else kv.contiguous()
    qbs = 0 if q.dim() == 2 else q.stride(0)
    with torch.cuda.device(dev):
        out = torch.empty((batches, n_q, C_), dtype=q.dtype, device=dev)
        _call('merv_cross_attention', lib.merv_cross_attention, q.data_ptr(), q.stride(-2), qbs, kv.data_ptr(), kv.stride(0), out.data_ptr(), C_,
              batches, n_q, n_kv, heads, hd, float(hd ** -0.5 if scale is None else scale), dtype_code(q.dtype), _stream())
    return out


def cross_attention_backward(q: torch.Tensor, kv: torch.Tensor, dout: torch.Tensor, batches: int, heads: int,
                             scale: Optional[float] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Gradients of `cross_attention`, fp32 or bf16, on every shape it runs: returns (dq [batches, n_q, C] — one dQ per batch entry, to
    be summed by the caller when the queries are shared — and dkv [batches * n_kv, 2C] = [dK | dV]) in the input dtype.  bf16 frames
    inside the tcgen05 tile take the tensor-core kernel, everything else the CUDA-core one (merv_cross_attention_backward_ex)."""
    lib = _lib.load()
    dev = _require_cuda(q, kv, dout)
    C_ = q.shape[-1]
    dt = q.dtype
    assert dt in (torch.float32, torch.bfloat16) and kv.dtype == dt and dout.dtype == dt
    assert kv.dim() == 2 and kv.shape[1] == 2 * C_ and kv.shape[0] % max(batches, 1) == 0 and C_ % heads == 0
    n_q, n_kv, hd = q.shape[-2], kv.shape[0] // max(batches, 1), C_ // heads
    assert dout.shape == (batches, n_q, C_)
    q = q if q.stride(-1) == 1 else q.contiguous()
    kv = kv if kv.stride(1) == 1 else kv.contiguous()
    dout = dout.contiguous()
    qbs = 0 if q.dim() == 2 else q.stride(0)
    code = dtype_code(dt)
    with torch.cuda.device(dev):
        dq = torch.empty((batches, n_q, C_), dtype=dt, device=dev)
        dkv = torch.empty((batches * n_kv, 2 * C_), dtype=dt, device=dev)
        n = lib.merv_cross_attention_backward_ex_workspace(batches, n_q, n_kv, heads, hd, code)
        ws = torch.empty(n, dtype=torch.float32, device=dev) if n else None
        _call('merv_cross_attention_backward_ex', lib.merv_cross_attention_backward_ex, q.data_ptr(), q.stride(-2), qbs, kv.data_ptr(),
              kv.stride(0), dout.data_ptr(), dout.stride(1), dq.data_ptr(), dq.stride(1), dkv.data_ptr(), dkv.stride(0), batches, n_q, n_kv,
              heads, hd, float(hd ** -0.5 if scale is None else scale), code, _p(ws), n, _stream())
    return dq, dkv


def add_rows(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a [M, C] + b [period, C] broadcast over row blocks (row m gets b[m % period]); period == M is a plain sum."""
    lib = _lib.load()
    dev = _require_cuda(a, b)
    assert a.dim() == 2 and b.dim() == 2 and a.shape[1] == b.shape[1] and a.dtype == b.dtype and a.shape[0] % b.shape[0] == 0
    a = a if a.stride(1) == 1 else a.contiguous()
    b = b if b.stride(1) == 1 else b.contiguous()
    with torch.cuda.device(dev):
        out = torch.empty(a.shape, dtype=a.dtype, device=dev)
        _call('merv_add_rows', lib.merv_add_rows, a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), out.data_ptr(), out.stride(0), a.shape[0],
              a.shape[1], b.shape[0], dtype_code(a.dtype), _stream())
    return out


def video_colsum(x: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """out[b, k] = scale * sum_t x[b, t, k] (fp32 [B, K]) for x [B, T, K]."""
    lib = _lib.load()
    dev = _require_cuda(x)
    assert x.dim() == 3
    x = _rows_in_place(x)
    B, T, K = x.shape
    with torch.cuda.device(dev):
        out = torch.empty((B, K), dtype=torch.float32, device=dev)
        _call('merv_video_colsum', lib.merv_video_colsum, x.data_ptr(), out.data_ptr(), B, T, K, x.stride(1), x.stride(0), float(scale),
              dtype_code(x.dtype), _stream())
    return out


def pair_dot(x: torch.Tensor, y: torch.Tensor, scale: Optional[torch.Tensor] = None):
    """Fixed-order partial sums [B, chunks] of sum_i x[b, i] * y[b, i] for x, y [B, ...] of equal shape.

    With ``scale`` (fp32 [B], any stride) also returns ``scale[b] * y[b]`` (shape of y) written in the same pass: the per-video mixing
    weight applied to the pooled tokens, the W-operand of the fused backward's dW GEMM."""
    lib = _lib.load()
    dev = _require_cuda(x, y, scale)
    assert x.shape == y.shape and x.dtype == y.dtype
    B = x.shape[0]
    shape = y.shape
    x, y = x.reshape(B, -1).contiguous(), y.reshape(B, -1).contiguous()
    with torch.cuda.device(dev):
        out = torch.empty((B, lib.merv_pair_dot_chunks()), dtype=torch.float32, device=dev)
        if scale is None:
            _call('merv_pair_dot', lib.merv_pair_dot, x.data_ptr(), y.data_ptr(), out.data_ptr(), B, x.shape[1], dtype_code(x.dtype), _stream())
            return out
        assert scale.dtype == torch.float32 and scale.dim() == 1 and scale.numel() == B
        ys = torch.empty_like(y)
        _call('merv_pair_dot', lib.merv_pair_dot_scale, x.data_ptr(), y.data_ptr(), out.data_ptr(), scale.data_ptr(), scale.stride(0), ys.data_ptr(), B,
              x.shape[1], dtype_code(x.dtype), _stream())
    return out, ys.view(shape)


def wgrad_video(dy: torch.Tensor, x: torch.Tensor, scale: torch.Tensor, w: torch.Tensor, videos: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """(dW [N_out, C] = sum_b scale[b] dy[b]^T x[b],  partials [videos, pair_dot_chunks] of <w, dy[b]^T x[b]>) in ONE tcgen05 pass over
    dy [videos * T, N_out] and x [videos * T, C], both read in place (include/merv_fusion.h: merv_wgrad_video).  `scale` fp32 [videos] (any
    stride), w [N_out, C] bf16.  T % 64 == 0.  dy may also be a [videos, T, N_out] view with any row / batch stride (the gradient of the prefix
    slot of the multimodal embedding buffer): read in place when TMA can address it (merv_wgrad_video_ex), otherwise copied."""
    lib = _lib.load()
    dev = _require_cuda(dy, x, scale, w)
    assert dy.dtype == x.dtype == w.dtype == torch.bfloat16 and scale.dtype == torch.float32 and scale.dim() == 1 and scale.numel() == videos
    if dy.dim() == 3:
        assert dy.shape[0] == videos
        dy = _rows_in_place(dy)
        lddy, dy_bs = dy.stride(1), dy.stride(0)
        dy2 = dy.shape[1] * videos, dy.shape[2]
    else:
        assert dy.dim() == 2 and dy.stride(1) == 1 and dy.shape[0] % videos == 0
        lddy, dy_bs = dy.stride(0), (dy.shape[0] // videos) * dy.stride(0)
        dy2 = tuple(dy.shape)
    assert x.dim() == 2 and dy2[0] == x.shape[0]
    assert x.stride(1) == 1 and w.stride(1) == 1 and w.shape == (dy2[1], x.shape[1])
    T = dy2[0] // videos
    N_out, Cc = w.shape
    with torch.cuda.device(dev):
        dW = torch.empty((N_out, Cc), dtype=torch.bfloat16, device=dev)
        partial = torch.empty((videos, lib.merv_pair_dot_chunks()), dtype=torch.float32, device=dev)
        ws = torch.empty(max(int(lib.merv_wgrad_video_workspace(videos, N_out, Cc)), 4), dtype=torch.float32, device=dev)
        _call('merv_wgrad_video', lib.merv_wgrad_video_ex, dy.data_ptr(), lddy, dy_bs, x.data_ptr(), x.stride(0), scale.data_ptr(), scale.stride(0),
              w.data_ptr(), w.stride(0), dW.data_ptr(), dW.stride(0), partial.data_ptr(), ws.data_ptr(), videos, T, N_out, Cc, _stream())
    return dW, partial


def fused_backward(weights: torch.Tensor, dweights_out: Optional[torch.Tensor], u: torch.Tensor, gsum: torch.Tensor,
                   dw_partials: Sequence[torch.Tensor], pbars: Sequence[torch.Tensor], Ws: Sequence[torch.Tensor],
                   biases: Sequence[Optional[torch.Tensor]], Q: torch.Tensor, Wq: torch.Tensor, Wk: torch.Tensor,
                   in_proj_bias: Optional[torch.Tensor], dWs: Sequence[torch.Tensor]):
    """Everything of the fused path's backward after its GEMMs (include/merv_fusion.h: merv_fused_backward).

    dWs[e] holds dOut^T (w_e (.) P_e) on entry and receives the rank-1 term u (x) g_e in place.
    Returns (ds [B, E] fp32, [db_e], dQ [1, embed], dWq, dWk, dbias [3 * embed]) in the compute dtype."""
    lib = _lib.load()
    dev = _require_cuda(weights, dweights_out, u, gsum, *dw_partials, *pbars, *Ws, *biases, Q, Wq, Wk, in_proj_bias, *dWs)
    B, E = weights.shape
    K = u.numel()
    embed = Wk.shape[0]
    dt = Ws[0].dtype
    assert weights.dtype == torch.float32 and weights.is_contiguous() and u.dtype == torch.float32 and gsum.shape == (B, K)
    assert dweights_out is None or (dweights_out.dtype == torch.float32 and dweights_out.is_contiguous() and dweights_out.shape == (B, E))
    assert all(w.stride(1) == 1 and w.dtype == dt for w in Ws) and all(d.stride(1) == 1 and d.dtype == dt for d in dWs)
    assert all(t.is_contiguous() for t in (Q, Wq, Wk)) and (in_proj_bias is None or in_proj_bias.is_contiguous())
    d = _lib.FusedBwdDesc()
    d.B, d.E, d.K, d.embed = B, E, K, embed
    with torch.cuda.device(dev):
        ds = torch.empty((B, E), dtype=torch.float32, device=dev)
        dbs = [torch.empty(K, dtype=dt, device=dev) if b is not None else None for b in biases]
        dQ = torch.empty((1, embed), dtype=dt, device=dev)
        dWq = torch.empty((embed, embed), dtype=dt, device=dev)
        dWk = torch.empty((embed, K), dtype=dt, device=dev)
        dbias = torch.empty(3 * embed, dtype=dt, device=dev)
        for e in range(E):
            d.C[e] = Ws[e].shape[1]
            assert dw_partials[e].is_contiguous() and pbars[e].is_contiguous() and pbars[e].shape == (B, Ws[e].shape[1]) and dWs[e].shape == Ws[e].shape
            d.dw_partial[e], d.pbar[e] = dw_partials[e].data_ptr(), pbars[e].data_ptr()
            d.W[e], d.ldw[e], d.bias[e] = Ws[e].data_ptr(), Ws[e].stride(0), _p(biases[e])
            d.dW[e], d.lddw[e], d.db[e] = dWs[e].data_ptr(), dWs[e].stride(0), _p(dbs[e])
        d.weights, d.dweights_out, d.u, d.gsum = weights.data_ptr(), _p(dweights_out), u.data_ptr(), gsum.data_ptr()
        d.Q, d.Wq, d.Wk, d.in_proj_bias = Q.data_ptr(), Wq.data_ptr(), Wk.data_ptr(), _p(in_proj_bias)
        d.ds, d.dQ, d.dWq, d.dWk, d.dbias = ds.data_ptr(), dQ.data_ptr(), dWq.data_ptr(), dWk.data_ptr(), dbias.data_ptr()
        n = lib.merv_fused_backward_workspace(C.byref(d))
        ws = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
        d.workspace, d.workspace_floats = ws.data_ptr(), n
        _call('merv_fused_backward', lib.merv_fused_backward, C.byref(d), dtype_code(dt), _stream())
    return ds, dbs, dQ, dWq, dWk, dbias


def gelu(z: torch.Tensor, dy: Optional[torch.Tensor] = None) -> torch.Tensor:
    """gelu(z) (exact erf), or dy * gelu'(z) when `dy` is given."""
    lib = _lib.load()
    dev = _require_cuda(z, dy)
    z = z.contiguous()
    dy = None if dy is None else dy.contiguous()
    with torch.cuda.device(dev):
        out = torch.empty_like(z)
        _call('merv_gelu', lib.merv_gelu, z.data_ptr(), _p(dy), out.data_ptr(), z.numel(), dtype_code(z.dtype), _stream())
    return out


def colsum(x: torch.Tensor) -> torch.Tensor:
    """sum over rows of [M, N] -> [N] in x.dtype (fp32 accumulation, fixed order)."""
    lib = _lib.load()
    dev = _require_cuda(x)
    assert x.dim() == 2 and x.stride(1) == 1
    M, N = x.shape
    with torch.cuda.device(dev):
        out = torch.empty(N, dtype=x.dtype, device=dev)
        ws = torch.empty(max(1, lib.merv_colsum_workspace(M, N)), dtype=torch.float32, device=dev)
        _call('merv_colsum', lib.merv_colsum, x.data_ptr(), out.data_ptr(), ws.data_ptr(), M, N, x.stride(0), dtype_code(x.dtype), _stream())
    return out


def mix_backward(Vs: Sequence[torch.Tensor], dout: torch.Tensor, weights: torch.Tensor, dweights: Optional[torch.Tensor], u: torch.Tensor,
                 Q: torch.Tensor, Wq: torch.Tensor, Wk: torch.Tensor, in_proj_bias: torch.Tensor):
    """Gradients of the adapter: returns (dV list, dQ [1, embed], dWq, dWk, d in_proj_bias) in the compute dtype."""
    lib = _lib.load()
    dev = _require_cuda(*Vs, dout, weights, dweights, u, Q, Wq, Wk, in_proj_bias)
    B, T, K = Vs[0].shape
    E, embed = len(Vs), Wk.shape[0]
    dt = Vs[0].dtype
    Vs = [v.contiguous() for v in Vs]
    dout = _rows_in_place(dout)
    assert all(v.shape == (B, T, K) and v.dtype == dt for v in Vs) and dout.shape == (B, T, K) and dout.dtype == dt
    assert weights.dtype == torch.float32 and weights.is_contiguous() and (dweights is None or (dweights.dtype == torch.float32 and dweights.is_contiguous()))
    with torch.cuda.device(dev):
        dVs = [torch.empty_like(v) for v in Vs]
        dQ = torch.empty((1, embed), dtype=dt, device=dev)
        dWq = torch.empty((embed, embed), dtype=dt, device=dev)
        dWk = torch.empty((embed, K), dtype=dt, device=dev)
        dbias = torch.empty(3 * embed, dtype=dt, device=dev)
        n = lib.merv_mix_backward_workspace(B, E, T, K, embed)  # every encoder at T tokens: no single-token column sums
        ws = torch.empty(n, dtype=torch.float32, device=dev)
        _call('merv_mix_backward', lib.merv_mix_backward_strided, ptr_array([v.data_ptr() for v in Vs]), i32_array([T] * E), dout.data_ptr(),
              dout.stride(1), dout.stride(0), weights.data_ptr(), _p(dweights), u.data_ptr(), 0, None, 0, Q.contiguous().data_ptr(),
              Wq.contiguous().data_ptr(), Wk.contiguous().data_ptr(), in_proj_bias.data_ptr(),
              ptr_array([d.data_ptr() for d in dVs]), dQ.data_ptr(), dWq.data_ptr(), dWk.data_ptr(), dbias.data_ptr(), None, ws.data_ptr(), n,
              B, E, T, K, embed, dtype_code(dt), _stream())
    return dVs, dQ, dWq, dWk, dbias


def mix_backward_ex(Vs: Sequence[torch.Tensor], dout: torch.Tensor, weights: torch.Tensor, dweights: Optional[torch.Tensor], u: torch.Tensor,
                    Q: torch.Tensor, Wq: torch.Tensor, Wk: torch.Tensor, in_proj_bias: torch.Tensor, per_token_u: bool = False,
                    pe: Optional[torch.Tensor] = None):
    """Gradients of the adapter in every configuration of its forward: V_e [B, T_e, K] with T_e in {T, 1} (dout is [B, T, K]),
    ``per_token_u`` for averagetoken=False (u and the rows of Wk are [T*K]), ``pe`` [E, K] for positional_embedding=True.
    Returns (dV list with each encoder's own T_e, dQ [1, embed], dWq, dWk, d in_proj_bias, dpe or None) in the compute dtype."""
    lib = _lib.load()
    dev = _require_cuda(*Vs, dout, weights, dweights, u, Q, Wq, Wk, in_proj_bias, pe)
    B, T, K = dout.shape
    E, embed = len(Vs), Wk.shape[0]
    dt = Vs[0].dtype
    Ku = T * K if per_token_u else K
    Vs = [v.contiguous() for v in Vs]
    dout = _rows_in_place(dout)
    assert all(v.shape in ((B, T, K), (B, 1, K)) and v.dtype == dt for v in Vs) and dout.dtype == dt
    assert u.dtype == torch.float32 and u.is_contiguous() and u.numel() == Ku and Wk.shape[1] == Ku
    assert weights.dtype == torch.float32 and weights.is_contiguous() and (dweights is None or (dweights.dtype == torch.float32 and dweights.is_contiguous()))
    assert pe is None or (not per_token_u and pe.shape == (E, K) and pe.dtype == dt)
    if pe is not None and pe.stride(1) != 1:
        pe = pe.contiguous()
    with torch.cuda.device(dev):
        dVs = [torch.empty_like(v) for v in Vs]
        dQ = torch.empty((1, embed), dtype=dt, device=dev)
        dWq = torch.empty((embed, embed), dtype=dt, device=dev)
        dWk = torch.empty((embed, Ku), dtype=dt, device=dev)
        dbias = torch.empty(3 * embed, dtype=dt, device=dev)
        dpe = None if pe is None else torch.empty((E, K), dtype=dt, device=dev)
        n = lib.merv_mix_backward_ex_workspace(B, E, T, K, embed, K if per_token_u else 0)
        ws = torch.empty(n, dtype=torch.float32, device=dev)
        _call('merv_mix_backward_ex', lib.merv_mix_backward_strided, ptr_array([v.data_ptr() for v in Vs]), i32_array([v.shape[1] for v in Vs]),
              dout.data_ptr(), dout.stride(1), dout.stride(0), weights.data_ptr(), _p(dweights), u.data_ptr(), K if per_token_u else 0, _p(pe), 0 if pe is None else pe.stride(0),
              Q.contiguous().data_ptr(), Wq.contiguous().data_ptr(), Wk.contiguous().data_ptr(), in_proj_bias.data_ptr(),
              ptr_array([d.data_ptr() for d in dVs]), dQ.data_ptr(), dWq.data_ptr(), dWk.data_ptr(), dbias.data_ptr(), _p(dpe), ws.data_ptr(), n,
              B, E, T, K, embed, dtype_code(dt), _stream())
    return dVs, dQ, dWq, dWk, dbias, dpe


def scalar_mix_backward(Vs: Sequence[torch.Tensor], dout: torch.Tensor, weights: torch.Tensor, dweights: Optional[torch.Tensor] = None):
    """Gradients of ScalarAdapter.forward (include/merv_fusion.h: merv_scalar_mix_backward): V_e and dout [B, T, K] of one shape and dtype,
    ``weights`` = softmax(scalar) fp32 [E], ``dweights`` fp32 [E] or None (gradient w.r.t. the returned weights).
    Returns (dV list in the dtype of V, dscalar fp32 [E])."""
    lib = _lib.load()
    dev = _require_cuda(*Vs, dout, weights, dweights)
    B, T, K = dout.shape
    E, dt = len(Vs), dout.dtype
    Vs = [v.contiguous() for v in Vs]
    dout = _rows_in_place(dout)
    assert all(v.shape == (B, T, K) and v.dtype == dt for v in Vs), "every encoder must have the [B, T, K] shape and dtype of dout"
    assert weights.dtype == torch.float32 and weights.is_contiguous() and weights.numel() == E
    assert dweights is None or (dweights.dtype == torch.float32 and dweights.is_contiguous() and dweights.numel() == E)
    with torch.cuda.device(dev):
        dVs = [torch.empty_like(v) for v in Vs]
        dscalar = torch.empty(E, dtype=torch.float32, device=dev)
        n = lib.merv_scalar_mix_backward_workspace(B, E, K)
        ws = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
        _call('merv_scalar_mix_backward', lib.merv_scalar_mix_backward_strided, ptr_array([v.data_ptr() for v in Vs]), dout.data_ptr(), dout.stride(1),
              dout.stride(0), weights.data_ptr(),
              _p(dweights), ptr_array([d.data_ptr() for d in dVs]), dscalar.data_ptr(), ws.data_ptr(), n, B, E, T, K, dtype_code(dt), _stream())
    return dVs, dscalar


def scalar_fused_backward(weights: torch.Tensor, dweights: Optional[torch.Tensor], gsum: torch.Tensor, dw_partials: Sequence[torch.Tensor],
                          biases: Sequence[Optional[torch.Tensor]]):
    """The end of the fused scalar training step (include/merv_fusion.h: merv_scalar_fused_backward): ``weights`` = softmax(scalar) fp32 [E],
    ``dweights`` fp32 [E] or None, ``gsum`` = video_colsum(dout) [B, K], ``dw_partials[e]`` from wgrad_video of encoder e, ``biases[e]`` [K].
    Returns (dscalar fp32 [E], [db_e] in the dtype of the biases)."""
    lib = _lib.load()
    dev = _require_cuda(weights, dweights, gsum, *dw_partials, *biases)
    B, K = gsum.shape
    E = weights.numel()
    present = [b for b in biases if b is not None]
    dt = present[0].dtype if present else torch.float32
    assert weights.dtype == torch.float32 and weights.is_contiguous() and gsum.dtype == torch.float32 and gsum.is_contiguous()
    assert dweights is None or (dweights.dtype == torch.float32 and dweights.is_contiguous() and dweights.numel() == E)
    assert len(dw_partials) == E and all(p.is_contiguous() and p.shape == (B, lib.merv_pair_dot_chunks()) for p in dw_partials)
    assert len(biases) == E and all(b.dtype == dt and b.is_contiguous() and b.numel() == K for b in present)
    with torch.cuda.device(dev):
        dscalar = torch.empty(E, dtype=torch.float32, device=dev)
        dbs = [None if b is None else torch.empty(K, dtype=dt, device=dev) for b in biases]
        n = lib.merv_scalar_fused_backward_workspace(E, K)
        ws = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
        _call('merv_scalar_fused_backward', lib.merv_scalar_fused_backward, weights.data_ptr(), _p(dweights), gsum.data_ptr(),
              ptr_array([p.data_ptr() for p in dw_partials]), ptr_array([_p(b) for b in biases]), ptr_array([_p(d) for d in dbs]), dscalar.data_ptr(),
              ws.data_ptr(), n, B, E, K, dtype_code(dt), _stream())
    return dscalar, dbs
