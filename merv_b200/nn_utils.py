"""B200-native drop-ins for the hot-path modules of the reference's ``merv/util/nn_utils.py``.

Same class names, constructor signatures, parameter names/shapes (hence state-dict keys), properties and
error behaviour as the reference (paths below are relative to the reference root):

    LinearProjector                      merv/util/nn_utils.py:22-32      (incl. pre_proj_layernorm)
    MLPProjector                         merv/util/nn_utils.py:35-59
    MLPDeepProjector                     merv/util/nn_utils.py:62-83
    FusedMLPProjector                    merv/util/nn_utils.py:86-108
    get_mlp_projector                    merv/util/nn_utils.py:111-121
    TokenResampler                       merv/util/nn_utils.py:124-133
    AveragePoolingProjector              merv/util/nn_utils.py:136-174    (2-D "avg")
    AttentivePooler (+ CrossAttention, MLP, CrossAttentionBlock containers)   merv/util/nn_utils.py:177-246,380-452  ("attntv", fp32 / bf16 training)
    AveragePooling3DProjector            merv/util/nn_utils.py:306-338
    Convolutional3DProjector             merv/util/nn_utils.py:341-377    ("3dconv": 27 displaced poolings + one GEMM on the pooled grid)
    CrossAttentionAdapterLearnableQuery  merv/util/nn_utils.py:455-521    (averagetoken either way, positional embedding)
    ScalarAdapter                        merv/util/nn_utils.py:524-537
    ConcatChannelFusion / ConcatChannelLNFusion                               merv/models/vidlms/merv.py:217-223,603-606

``forward`` runs hand-written sm_100a kernels through the C ABI (``merv_b200.ops``); nothing here calls a
torch compute op on the data path, and CPU tensors raise.  ``nn.Linear`` / ``nn.MultiheadAttention`` are used
purely as parameter containers so initialisation (RNG consumption order under ``torch.manual_seed``,
merv.py:87), ``state_dict`` keys and FSDP wrapping behave exactly like the reference.

Two execution modes:

* module-by-module (default): each projector returns its ``[B, T*S*S, llm_dim]`` tokens, the adapter scores,
  soft-maxes and mixes them — a drop-in for any caller of the individual modules;
* linked (``link_fused`` / ``MervFusion`` / ``patch_merv``): projectors return a ``DeferredProjection`` and the
  adapter runs the whole path as pool -> [hidden layers] -> scores -> ONE tcgen05 GEMM whose epilogue applies the
  mixing weights, so the per-encoder projections never touch HBM.  Valid whenever the LAST projector layer is
  affine (true for every projector type of the reference).  In grad mode the linear projectors take the same fused
  forward with a backward that keeps only the pooled tokens (``_FusedLinearFn``, or ``_FusedScalarLinearFn`` in front of the
  scalar mixer) unless FSDP manages a parameter involved; everything else trains through the module-by-module autograd Functions.
"""

from __future__ import annotations

import math
import weakref
from abc import ABC, abstractmethod
from typing import List, Optional, Sequence, Tuple, Union

import torch
import torch.nn as nn
from torch.nn.init import xavier_uniform_
from torch.nn.parameter import Parameter

from . import ops
from ._lib import ACT_GELU_ERF, ACT_NONE, MAX_SEGMENTS

IGNORE_INDEX = -100  # merv.py:53


# ------------------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------------------
def _compute_dtype(x: torch.Tensor) -> torch.dtype:
    """bf16 under torch.autocast('cuda', bfloat16) (merv.py:816, base_strategy.py:210-214), else the input dtype."""
    if torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
        if dt != torch.bfloat16:
            raise TypeError(f"merv_b200 supports bf16 autocast only, got {dt}")
        return dt
    if x.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError(f"merv_b200 supports float32 and bfloat16, got {x.dtype}")
    return x.dtype


def _require_device(t: torch.Tensor) -> None:
    if not t.is_cuda:
        raise RuntimeError("merv_b200 runs only on CUDA (sm_100a) tensors; there is deliberately no CPU fallback.")


def _tma_readable(x: torch.Tensor) -> bool:
    """Feature tensor the pool kernel reads in place: channels contiguous, every other stride a multiple of one 16-byte vector
    (bf16), 16-byte aligned base — e.g. a CLS-dropping slice of a backbone output.  Anything else is copied first."""
    return x.stride(3) == 1 and not any(st % 8 for st in x.stride()[:3]) and x.data_ptr() % 16 == 0


def _as_batch_index(batch_index: Optional[torch.Tensor], like: torch.Tensor) -> Optional[torch.Tensor]:
    """`multimodal_indices` (merv.py:572; int64 in the reference) as the contiguous int32 device vector the kernels gather by."""
    if batch_index is None:
        return None
    assert batch_index.dim() == 1 and not batch_index.is_floating_point(), "batch_index must be a 1-D integer tensor"
    if batch_index.device != like.device or batch_index.dtype != torch.int32 or not batch_index.is_contiguous():
        batch_index = batch_index.to(device=like.device, dtype=torch.int32).contiguous()
    return batch_index


def _stream_key(dev: torch.device) -> Tuple[int, int]:
    """(device index, current stream handle): cached plans own workspaces, so they are bound to one stream."""
    return dev.index, torch.cuda.current_stream(dev).cuda_stream


def _is_sharded_param(p: torch.Tensor) -> bool:
    """Parameter managed by FSDP (flattened original parameter of FSDP1, DTensor of FSDP2): its full value only exists inside its own
    unit's forward / backward."""
    return bool(getattr(p, "_fsdp_flattened", False)) or hasattr(p, "_local_tensor") or type(p).__name__ == "FlatParameter"


def _needs_grad(module: nn.Module, *tensors) -> bool:
    """True when the call must be recorded by autograd (training step: projectors and adapter are trainable in every
    stage, merv.py:318-320,342-343,363-365)."""
    return torch.is_grad_enabled() and (
        any(p.requires_grad for p in module.parameters()) or any(isinstance(t, torch.Tensor) and t.requires_grad for t in tensors)
    )


def _linear_wgrad(g: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """dW = g^T x of a Linear (g [M, N], x [M, K] -> [N, K]), a contraction over the tokens.  bf16: the tensor cores read both operands
    MN-major in place; fp32 (the parity path, SIMT GEMM, K-major) transposes them first."""
    if g.dtype == torch.bfloat16:
        return ops.gemm_ex(g, x, a_t=True, w_t=True)
    dW, _ = ops.linear_bias_act(ops.transpose(g, pad=True), ops.transpose(x, pad=True), None, ACT_NONE)  # [N, M] x [K, M]^T
    return dW


def _linear_dgrad(g: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """dX = g W of a Linear (g [M, N], W [N, K] -> [M, K]); bf16 reads W MN-major in place, fp32 transposes it."""
    if g.dtype == torch.bfloat16:
        return ops.gemm_ex(g, w, w_t=True)
    dx, _ = ops.linear_bias_act(g, ops.transpose(w), None, ACT_NONE)  # [M, N] x [K, N]^T
    return dx


class _ProjectorFn(torch.autograd.Function):
    """[LayerNorm ->] Linear / gelu-mlp / fused-gelu-mlp projector (nn_utils.py:22-108) with a hand-written backward.

    forward : X_0 = LN(x) (pre_proj_layernorm) or x;  Z_i = X_i W_i^T + b_i on the sm_100a GEMM (pre-activations kept),
              X_{i+1} = gelu(Z_i)
    backward: dZ_i = dX_{i+1} * gelu'(Z_i);  dW_i = dZ_i^T X_i and dX_i = dZ_i W_i (same GEMM on transposed copies — the
              kernel is K-major);  db_i = colsum(dZ_i);  LayerNorm: dgamma = colsum(dX_0 * xhat), dbeta = colsum(dX_0)
    The gradient w.r.t. the input is produced only when the input requires it (projected tokens entering the
    concat_channel fusion); the patch features never do: the backbones are frozen (merv.py:316,339,361).
    """

    @staticmethod
    def forward(ctx, x, acts, dtype, cache, ln_eps, *params):
        # params = ([gamma, beta,] W_0, b_0, W_1, b_1, ...) — the nn.Parameters, so autograd routes the gradients;
        # compute-dtype copies come from `cache`
        has_ln = ln_eps is not None
        lin_params = params[2:] if has_ln else params
        n = len(acts)
        x_in, gamma = x, None
        if has_ln:
            gamma = cache.get(params[0], dtype)
            x = ops.layernorm([x], gamma, cache.get(params[1], dtype), ln_eps)
        xs, zs, ws = [x], [], []
        for i in range(n):
            w_c, b_c = cache.get(lin_params[2 * i], dtype), cache.get(lin_params[2 * i + 1], dtype)
            z, _ = ops.linear_bias_act(xs[-1], w_c, b_c, ACT_NONE)
            ws.append(w_c)
            if acts[i] == ACT_GELU_ERF:
                zs.append(z)
                xs.append(ops.gelu(z))
            else:
                zs.append(None)
                xs.append(z)
        ctx.acts = acts
        ctx.param_dtypes = [p.dtype for p in params]
        ctx.nz = [z is not None for z in zs]
        ctx.ln_eps = ln_eps
        ctx.save_for_backward(*xs[:-1], *[z for z in zs if z is not None], *ws, *([x_in, gamma] if has_ln else []))
        return xs[-1]

    @staticmethod
    def backward(ctx, dy):
        n = len(ctx.acts)
        has_ln = ctx.ln_eps is not None
        saved = list(ctx.saved_tensors)
        xs = saved[:n]
        nz = sum(ctx.nz)
        z_it = iter(saved[n:n + nz])
        zs = [next(z_it) if has else None for has in ctx.nz]
        ws = saved[n + nz:n + nz + n]
        need_dx = ctx.needs_input_grad[0]
        g = dy.reshape(-1, dy.shape[-1])
        if g.dtype != xs[0].dtype:
            g = g.to(xs[0].dtype)
        if g.stride(1) != 1:
            g = g.contiguous()
        off = 2 if has_ln else 0
        grads = [None] * (2 * n + off)
        for i in reversed(range(n)):
            if zs[i] is not None:
                g = ops.gelu(zs[i].reshape(g.shape), g)  # dZ_i
            dW = _linear_wgrad(g, xs[i].reshape(-1, xs[i].shape[-1]))  # dW_i = dZ_i^T X_i
            grads[off + 2 * i] = dW.to(ctx.param_dtypes[off + 2 * i])
            grads[off + 2 * i + 1] = ops.colsum(g).to(ctx.param_dtypes[off + 2 * i + 1])
            if i > 0 or need_dx or has_ln:
                g = _linear_dgrad(g, ws[i])  # dX_i = dZ_i W_i
        dx = g if need_dx else None
        if has_ln:
            x_in, gamma = saved[-2], saved[-1]
            dx, dgamma, dbeta = ops.layernorm_backward([x_in], g, gamma, ctx.ln_eps, need_dx=need_dx)
            grads[0], grads[1] = dgamma.to(ctx.param_dtypes[0]), dbeta.to(ctx.param_dtypes[1])
        if dx is not None:
            dx = dx.reshape(xs[0].shape)
        return (dx, None, None, None, None, *grads)


class _ConvTapsFn(torch.autograd.Function):
    """pool(conv3d(x)) as ONE GEMM over the 27 pooled taps (Convolutional3DProjector.convolution_pooling, nn_utils.py:349-352,364).

    forward : Y = A W2^T + b with A [M, 27 C] = ops.pool3d_conv_taps(x) and W2 [K, 27 C] the tap-major view of the Conv3d weight
    backward: dW2 = dY^T A (tensor cores read both operands MN-major in place), db = colsum(dY); nothing flows into the patch features
              (frozen backbones, merv.py:316,339,361)."""

    @staticmethod
    def forward(ctx, A, dtype, module, weight, bias):
        W2, b = module._conv_operands(dtype)
        y, _ = ops.linear_bias_act(A, W2, b, ACT_NONE)
        ctx.save_for_backward(A)
        ctx.wshape, ctx.wdtype, ctx.bdtype = tuple(weight.shape), weight.dtype, None if bias is None else bias.dtype
        return y

    @staticmethod
    def backward(ctx, dy):
        (A,) = ctx.saved_tensors
        A2 = A.reshape(-1, A.shape[-1])
        g = dy.reshape(-1, dy.shape[-1])
        if g.dtype != A2.dtype:
            g = g.to(A2.dtype)
        if g.stride(1) != 1:
            g = g.contiguous()
        dW2 = _linear_wgrad(g, A2)
        K, C = ctx.wshape[0], ctx.wshape[1]
        dW = dW2.reshape(K, 3, 3, 3, C).permute(0, 4, 1, 2, 3).to(ctx.wdtype)  # back to Conv3d's [K, C, kf, kh, kw]
        db = None if ctx.bdtype is None else ops.colsum(g).to(ctx.bdtype)
        return None, None, None, dW, db


class _Assembly:
    """MERV.forward's ``[BOS | prefix | text]`` assembly (merv.py:622-720) done INSIDE a mixer's autograd Function, which then owns the whole
    embedding buffer: the kernels write the prefix into its slot and its backward reads the prefix gradient from the buffer's gradient in place.
    (An in-place write into a view of a buffer autograd tracks would make CopySlices clone the whole gradient: the copy this avoids.)

    Rows ``idx`` (multimodal) come first as [BOS | prefix | text], then rows ``uni`` (text only) padded at the end with T zero rows.
    ``emb`` [Bt, L, K] is the text embedding tensor; it is one more differentiable input of the Function."""

    def __init__(self, emb: torch.Tensor, idx: torch.Tensor, uni: torch.Tensor, bos: int) -> None:
        self.emb, self.idx, self.uni, self.bos = emb, idx, uni, bos

    def buffer(self, T: int, K: int, dtype: torch.dtype) -> Tuple[torch.Tensor, torch.Tensor]:
        """(buf [Bm + Bu, L + T, K] in `dtype` with the text spliced in, its prefix slot buf[:Bm, bos:bos + T])."""
        e, idx, uni, bos = self.emb.detach(), self.idx, self.uni, self.bos
        Bm, Bu, L = idx.numel(), uni.numel(), e.shape[1]
        assert e.shape[2] == K, f"input_embeddings have {e.shape[2]} channels, the prefix {K}"
        buf = torch.empty((Bm + Bu, L + T, K), dtype=dtype, device=e.device)
        buf[:Bm, :bos].copy_(e[idx, :bos])
        buf[:Bm, bos + T:].copy_(e[idx, bos:])
        if Bu:
            buf[Bm:, :L].copy_(e[uni])
            buf[Bm:, L:].zero_()
        return buf, buf[:Bm, bos:bos + T]

    def grads(self, dbuf: Optional[torch.Tensor], T: int, dtype: torch.dtype, need_emb: bool):
        """(prefix-slot gradient [Bm, T, K], a view of dbuf unless dbuf had to be made contiguous in `dtype`; d input_embeddings or None).
        The text parts of dbuf go back to rows idx / uni; rows in neither set get zeros."""
        idx, uni, bos = self.idx, self.uni, self.bos
        Bm, L = idx.numel(), self.emb.shape[1]
        if dbuf is None:  # only the mixing weights were used downstream
            return None, None
        if dbuf.dtype != dtype or not dbuf.is_contiguous():
            dbuf = dbuf.to(dtype).contiguous()
        demb = None
        if need_emb:
            demb = torch.zeros(self.emb.shape, dtype=self.emb.dtype, device=dbuf.device)
            demb.index_add_(0, idx, torch.cat([dbuf[:Bm, :bos], dbuf[:Bm, bos + T:]], 1).to(demb.dtype))
            if uni.numel():
                demb.index_add_(0, uni, dbuf[Bm:, :L].to(demb.dtype))
        return dbuf[:Bm, bos:bos + T], demb


class _MixFn(torch.autograd.Function):
    """CrossAttentionAdapterLearnableQuery.forward (nn_utils.py:487-521) with its hand-written backward, in every configuration:
    averagetoken=True / False, single-token (repeated) encoders, and positional_embedding=True, where ``pe`` is an input (None
    otherwise: with averagetoken=False the reference never reads it, so it gets no gradient).  With an assembly (``asm``, see _Assembly) the
    fused tokens go into the prefix slot of the embedding buffer, which is returned instead, and ``emb`` gets its gradient."""

    @staticmethod
    def forward(ctx, adapter, dtype, asm, emb, Q, Wq, Wk, bias, pe, *V):
        c = adapter._cast_cache
        Vc = [v if v.dtype == dtype else v.to(dtype) for v in V]
        u = adapter.query_vector(dtype)  # [K], or [T*K] with averagetoken=False (the key is the flattened token block)
        per_token_u = not adapter.averagetoken
        T = adapter.token_length
        scores = ops.scores_from_tokens(Vc, u, T, per_token_u=per_token_u, consts=adapter._pe_consts(dtype), mean=adapter.averagetoken)
        buf, slot = (None, None) if asm is None else asm.buffer(T, Vc[0].shape[2], dtype)
        if slot is None:
            out, weights = ops.softmax_mix(Vc, T, scores=scores)
        else:
            _, weights = ops.softmax_mix(Vc, T, scores=scores, out=slot)
        params = (Q, Wq, Wk, bias) + (() if pe is None else (pe,))
        ctx.save_for_backward(weights, u, *[c.get(p, dtype) for p in params], *Vc)
        ctx.meta = (dtype, per_token_u, [p.dtype for p in params], [v.dtype for v in V])
        ctx.asm, ctx.T = asm, T
        return (out if asm is None else buf), weights.to(dtype)

    @staticmethod
    def backward(ctx, dout, dweights):
        dtype, per_token_u, pdt, vdt = ctx.meta
        weights, u, Qc, Wqc, Wkc, bc, *rest = ctx.saved_tensors
        pec, Vc = (rest[0], rest[1:]) if len(pdt) == 5 else (None, rest)
        demb = None
        if ctx.asm is not None:  # the prefix slot of the buffer's gradient, read in place by the kernels
            dout, demb = ctx.asm.grads(dout, ctx.T, dtype, ctx.needs_input_grad[3])
        if dout is None:  # only the mixing weights were used downstream
            dout = torch.zeros((weights.shape[0], ctx.T, Vc[0].shape[2]), dtype=dtype, device=weights.device)
        dw = None if dweights is None else dweights.float().contiguous()
        if per_token_u or pec is not None or any(v.shape[1] != dout.shape[1] for v in Vc):
            dVs, dQ, dWq, dWk, dbias, dpe = ops.mix_backward_ex(Vc, dout.to(dtype), weights, dw, u, Qc, Wqc, Wkc, bc, per_token_u=per_token_u, pe=pec)
        else:  # the configuration MERV constructs (merv.py:214-216): the same kernels, bit-identical to mix_backward_ex
            (dVs, dQ, dWq, dWk, dbias), dpe = ops.mix_backward(Vc, dout.to(dtype), weights, dw, u, Qc, Wqc, Wkc, bc), None
        grads = [g.to(t) for g, t in zip((dQ, dWq, dWk, dbias, dpe), pdt)]
        if dpe is None:
            grads.append(None)
        return (None, None, None, demb, *grads, *[g.to(t) for g, t in zip(dVs, vdt)])


class _ScalarMixFn(torch.autograd.Function):
    """ScalarAdapter.forward (nn_utils.py:524-537) with its hand-written backward: w = softmax(scalar) [E] for every video,
    out = sum_e w_e V_e, returns (out, w[None]).  dV_e = w_e dOut and dscalar = w (.) (g - <w, g>) with
    g_e = sum_b <dOut[b], V_e[b]> + dW_out[e], in one pass over dOut and the V_e (merv_scalar_mix_backward).  Every V_e is [B, T, K]:
    the reference stacks them.  The scalar gradient comes back in the parameter's dtype (fp32 master weights under autocast).  With an
    assembly (``asm``, see _Assembly) the mix goes into the prefix slot of the embedding buffer, which is returned instead."""

    @staticmethod
    def forward(ctx, scalar, dtype, asm, emb, *V):
        Vc = [v if v.dtype == dtype else v.to(dtype) for v in V]
        B, T, K = Vc[0].shape
        E = len(Vc)
        w, _ = ops.softmax_weights(scalar.detach().float().reshape(1, E))
        buf, slot = (None, None) if asm is None else asm.buffer(T, K, dtype)
        if B > 0 and slot is not None:
            ops.softmax_mix(Vc, T, weights=w.expand(B, E).contiguous(), out=slot)
        elif B > 0:
            out, _ = ops.softmax_mix(Vc, T, weights=w.expand(B, E).contiguous())
        else:  # a rank that owns no videos (merv_b200/parallel.py): no mix to launch, the weights still carry a gradient
            out = torch.empty((0, T, K), dtype=dtype, device=Vc[0].device)
        ctx.save_for_backward(w, *Vc)
        ctx.meta = (scalar.dtype, [v.dtype for v in V])
        ctx.asm = asm
        return (out if asm is None else buf), w.to(dtype)

    @staticmethod
    def backward(ctx, dout, dweights):
        w, *Vc = ctx.saved_tensors
        sdt, vdt = ctx.meta
        dt = Vc[0].dtype
        demb = None
        if ctx.asm is not None:  # the prefix slot of the buffer's gradient, read in place by the kernel
            dout, demb = ctx.asm.grads(dout, Vc[0].shape[1], dt, ctx.needs_input_grad[3])
        if dout is None:  # only the mixing weights were used downstream
            dout = torch.zeros_like(Vc[0])
        dw = None if dweights is None else dweights.float().reshape(-1).contiguous()
        dVs, dscalar = ops.scalar_mix_backward(Vc, dout.to(dt), w.reshape(-1), dw)
        return (dscalar.to(sdt), None, None, demb, *[g.to(t) for g, t in zip(dVs, vdt)])


class _AttentivePoolFn(torch.autograd.Function):
    """AttentivePooler.forward up to (not including) its projector (nn_utils.py:229-237 with CrossAttentionBlock.forward :447-451 and
    CrossAttention.forward :393-412) in the compute dtype (fp32 or bf16), with a hand-written backward; the patch features get no
    gradient (frozen backbones).

    forward : xn = LN1(x);  kv = xn Wkv^T + bkv;  qp = qt Wq^T + bq;  a = attention(qp, kv);  y = a Wp^T + bp;  q1 = y + qt;
              hn = LN2(q1);  z1 = hn W1^T + b1;  g1 = gelu(z1);  h2 = g1 W2^T + b2;  q2 = q1 + h2
    backward: every Linear as dW = dY^T X and dX = dY W (_linear_wgrad / _linear_dgrad: the MN-major tcgen05 GEMM in bf16, the SIMT GEMM
              on transposed copies in fp32), the attention through merv_cross_attention_backward_ex (five tcgen05 contractions per frame
              and head for bf16 frames inside its tile, the CUDA-core kernel for every other shape and for fp32), LayerNorm / GELU /
              reductions through their HBM-bound kernels.  The learned queries are shared by all frames: their gradient sums the frames."""

    @staticmethod
    def forward(ctx, x, dtype, cache, heads, scale, eps1, eps2, qt3, g1w, g1b, Wkv, bkv, Wq, bq, Wp, bp, g2w, g2b, W1, b1, W2, b2):
        dt = dtype
        c = cache
        B, F, N, C_ = x.shape
        n = qt3.shape[1]
        xf = x.reshape(B * F * N, C_)
        P = [c.get(t, dt) for t in (qt3, g1w, g1b, Wkv, bkv, Wq, bq, Wp, bp, g2w, g2b, W1, b1, W2, b2)]
        qt3c, g1wc, g1bc, Wkvc, bkvc, Wqc, bqc, Wpc, bpc, g2wc, g2bc, W1c, b1c, W2c, b2c = P
        qt = qt3c[0]
        xn = ops.layernorm([xf], g1wc, g1bc, eps1)
        kv, _ = ops.linear_bias_act(xn, Wkvc, bkvc, ACT_NONE)
        qp, _ = ops.linear_bias_act(qt, Wqc, bqc, ACT_NONE)
        a = ops.cross_attention(qp, kv, B * F, heads, scale)
        a2 = a.view(B * F * n, C_)
        y, _ = ops.linear_bias_act(a2, Wpc, bpc, ACT_NONE)
        q1 = ops.add_rows(y, qt)
        hn = ops.layernorm([q1], g2wc, g2bc, eps2)
        z1, _ = ops.linear_bias_act(hn, W1c, b1c, ACT_NONE)
        g1 = ops.gelu(z1)
        h2, _ = ops.linear_bias_act(g1, W2c, b2c, ACT_NONE)
        q2 = ops.add_rows(q1, h2)
        ctx.meta = (heads, scale, eps1, eps2, (B, F, N, C_, n), [t.dtype for t in (qt3, g1w, g1b, Wkv, bkv, Wq, bq, Wp, bp, g2w, g2b, W1, b1, W2, b2)])
        ctx.save_for_backward(xf, xn, kv, qp, a2, q1, hn, z1, g1, qt, g1wc, Wkvc, Wqc, Wpc, g2wc, W1c, W2c)
        return q2

    @staticmethod
    def backward(ctx, dq2):
        heads, scale, eps1, eps2, (B, F, N, C_, n), pdt = ctx.meta
        xf, xn, kv, qp, a2, q1, hn, z1, g1, qt, g1wc, Wkvc, Wqc, Wpc, g2wc, W1c, W2c = ctx.saved_tensors
        dt = xf.dtype
        g = dq2.reshape(-1, C_)
        g = (g if g.dtype == dt else g.to(dt)).contiguous()
        BF = B * F
        # q2 = q1 + fc2(gelu(fc1(LN2(q1))))
        dW2 = _linear_wgrad(g, g1)
        db2 = ops.colsum(g)
        dz1 = ops.gelu(z1, _linear_dgrad(g, W2c))
        dW1 = _linear_wgrad(dz1, hn)
        db1 = ops.colsum(dz1)
        dq1_ln, dg2w, dg2b = ops.layernorm_backward([q1], _linear_dgrad(dz1, W1c), g2wc, eps2)
        dq1 = ops.add_rows(g, dq1_ln)
        # q1 = proj(attention) + query tokens (the same tokens for every frame)
        dqt = ops.video_colsum(dq1.view(1, BF, n * C_)).view(n, C_)  # fp32
        dWp = _linear_wgrad(dq1, a2)
        dbp = ops.colsum(dq1)
        da = _linear_dgrad(dq1, Wpc)
        dq_frames, dkv = ops.cross_attention_backward(qp, kv, da.view(BF, n, C_), BF, heads, scale)
        dqp = ops.video_colsum(dq_frames.view(1, BF, n * C_)).view(n, C_).to(dt)
        dWq = _linear_wgrad(dqp, qt)
        dbq = ops.colsum(dqp)
        dqt = dqt + _linear_dgrad(dqp, Wqc).float()
        dWkv = _linear_wgrad(dkv, xn)
        dbkv = ops.colsum(dkv)
        _, dg1w, dg1b = ops.layernorm_backward([xf], _linear_dgrad(dkv, Wkvc), g1wc, eps1, need_dx=False)
        grads = [dqt.view(1, n, C_), dg1w, dg1b, dWkv, dbkv, dWq, dbq, dWp, dbp, dg2w, dg2b, dW1, db1, dW2, db2]
        return (None, None, None, None, None, None, None, *[gr.to(t) for gr, t in zip(grads, pdt)])


def _version(p: torch.Tensor) -> int:
    """In-place-update counter of a parameter; inference tensors do not track one (and cannot be updated in place
    outside inference mode), so they count as version 0."""
    try:
        return p._version
    except RuntimeError:
        return 0


def _is_volatile(p: Optional[torch.Tensor]) -> bool:
    """A "parameter" that is not an ``nn.Parameter``: inside an FSDP1 unit's forward (``use_orig_params=True``, fsdp.py:240) the
    module attributes are fresh VIEWS into the unit's unsharded flat buffer.  That buffer keeps its address from step to step
    while the optimizer rewrites its contents through the sharded master copy, and a fresh view always reports ``_version`` 0 —
    so nothing derived from such a tensor may be cached on (data_ptr, version)."""
    return p is not None and not isinstance(p, nn.Parameter)


class _CastCache:
    """Weights cast to the compute dtype, keyed on (storage, version) so in-place optimiser updates invalidate them."""

    def __init__(self) -> None:
        self._store = {}

    def get(self, p: Optional[torch.Tensor], dtype: torch.dtype) -> Optional[torch.Tensor]:
        if p is None:
            return None
        if p.dtype == dtype and p.data_ptr() % 16 == 0 and p.is_contiguous():
            return p.detach()
        if _is_volatile(p):  # FSDP view: a new object with unknowable contents every forward — convert, never remember
            return p.detach().to(dtype).contiguous().clone() if p.dtype == dtype else p.detach().to(dtype).contiguous()
        # (a same-dtype parameter that is a misaligned / strided view — e.g. FSDP's use_orig_params views into a flat
        #  buffer, fsdp.py:240 — is copied once per version: TMA and the 128-bit loads need 16-byte aligned rows)
        key = (id(p), dtype)
        tag = (p.data_ptr(), _version(p), tuple(p.shape))
        hit = self._store.get(key)
        if hit is None or hit[0] != tag:
            hit = (tag, p.detach().to(dtype).contiguous().clone() if p.dtype == dtype else p.detach().to(dtype).contiguous())
            self._store[key] = hit
        return hit[1]


def _fused_mix_into(asm: Optional[_Assembly], pooled, Ws, weights, bias_mix, B: int, T: int, K: int):
    """The fused GEMM's prefix [B, T, K] and the embedding buffer (None without an assembly).  The GEMM stores straight into the buffer's
    prefix slot when T % 128 == 0 (its batch-strided store); otherwise the prefix is computed contiguous and copied in."""
    if asm is None:
        return ops.fused_linear_mix(pooled, Ws, weights, bias_mix, T).view(B, T, K), None
    buf, slot = asm.buffer(T, K, torch.bfloat16)
    if T % 128 == 0:
        ops.fused_linear_mix(pooled, Ws, weights, bias_mix, T, out=slot)
    else:
        slot.copy_(ops.fused_linear_mix(pooled, Ws, weights, bias_mix, T).view(B, T, K))
    return slot, buf


def _fused_dout(asm: Optional[_Assembly], dout, B: int, T: int, K: int, dt: torch.dtype, device, need_emb: bool):
    """(dOut [B, T, K] in `dt` — the prefix slot of the buffer's gradient, read in place — and d input_embeddings) for the fused backwards."""
    demb = None
    if asm is not None:
        dout, demb = asm.grads(dout, T, dt, need_emb)
    if dout is None:  # only the mixing weights were used downstream
        return torch.zeros((B, T, K), dtype=dt, device=device), demb
    if dout.dtype != dt:
        dout = dout.to(dt)
    if dout.stride(2) != 1:
        dout = dout.contiguous()
    # the videos' rows back to back: one [B * T, K] matrix, as the GEMMs took it before any embedding buffer existed
    return (dout.view(B * T, K) if dout.is_contiguous() else dout), demb


class _FusedLinearFn(torch.autograd.Function):
    """Training step of the shipped configuration (3d-avg pool + linear projectors + learnable-query mixer, merv.py:587-589,608)
    through the FUSED forward, with a backward that never materialises the per-encoder projections Y_e or their gradients.

    forward : merv_pool3d (+ score partials) -> scores -> softmax -> merv_fused_linear_mix; keeps the pooled tokens P_e and the weights
    backward: G_e[b] = dOut[b]^T P_e[b] on tcgen05, drained once per video:  dW_e = sum_b w_e[b] G_e[b] + u (x) g_e  and
              dw_e[b] = <W_e, G_e[b]> + b_e . colsum_t(dOut[b])  (= <dOut[b] W_e, P_e[b]> without the Z_e = dOut W_e GEMM: merv_wgrad_video);
              ds = softmax'(dw + dweights);  db_e, du -> dQ, dWq, dWk, db_q  (include/merv_fusion.h: merv_fused_backward).
              Token counts that are not a multiple of 64 take the two-GEMM form (Z_e = dOut W_e, dW_e = dOut^T (w_e (.) P_e)).
    Per video this moves ~100 MB less through HBM in the forward and ~130 MB less in the backward than the module-by-module
    path and keeps 7 MB instead of 41 MB of activations.  No gradient flows into the patch features (frozen backbones).
    ``batch_index`` gathers the videos inside the pool kernel (``multimodal_indices``); with an assembly (``asm``, see _Assembly) the GEMM
    writes the prefix into its slot of the embedding buffer (T % 128 == 0; otherwise it is computed contiguous and copied in), the buffer is
    returned, and the backward reads dOut from the buffer's gradient in place.
    """

    @staticmethod
    def forward(ctx, fusion, projs, xs, batch_index, asm, emb, Q, Wq, Wk, in_proj_bias, *proj_params):
        dtype = torch.bfloat16
        E = len(projs)
        T, K = fusion.token_length, fusion.llm_dim
        B = xs[0].shape[0] if batch_index is None else batch_index.numel()
        lasts = [p.layers()[-1][0] for p in projs]
        vcs = [fusion._affine_vec(lin, p._cast_cache, dtype) for lin, p in zip(lasts, projs)]
        Ws = [p._cast_cache.get(lin.weight, dtype) for lin, p in zip(lasts, projs)]
        biases = [p._cast_cache.get(lin.bias, dtype) for lin, p in zip(lasts, projs)]
        pooled, partials = fusion._fused_stage1(projs, xs, vcs, dtype, batch_index=batch_index)
        scores = ops.scores_from_partials(partials, [vc[1] for vc in vcs], B, T)
        weights, bias_mix = ops.softmax_weights(scores, biases, K)
        out, buf = _fused_mix_into(asm, pooled, Ws, weights, bias_mix, B, T, K)
        c = fusion._cast_cache
        ctx.fusion_dims = (B, E, T, K)
        ctx.asm = asm
        ctx.param_dtypes = [t.dtype for t in (Q, Wq, Wk, in_proj_bias, *proj_params)]
        ctx.save_for_backward(weights, fusion.query_vector(dtype), c.get(Q, dtype), c.get(Wq, dtype), c.get(Wk, dtype), c.get(in_proj_bias, dtype),
                              *pooled, *Ws, *biases)
        w_out = weights.to(dtype)
        return (out if asm is None else buf), w_out

    @staticmethod
    def backward(ctx, dout, dweights):
        B, E, T, K = ctx.fusion_dims
        saved = list(ctx.saved_tensors)
        weights, u, Qc, Wqc, Wkc, bc = saved[:6]
        pooled, Ws, biases = saved[6:6 + E], saved[6 + E:6 + 2 * E], saved[6 + 2 * E:6 + 3 * E]
        dt = Ws[0].dtype
        g, demb = _fused_dout(ctx.asm, dout, B, T, K, dt, weights.device, ctx.needs_input_grad[5])
        dwo = None if dweights is None else dweights.float().contiguous()
        gsum = ops.video_colsum(g.view(B, T, K))
        if T % 64:  # the two-GEMM form below reads dOut as one [B * T, K] matrix
            g = g.contiguous().view(B * T, K)
        dw_partials, pbars, dWs = [], [], []
        for e in range(E):  # dOut, P_e and W_e are all read in place: the tensor cores take them MN-major (no transposed copies)
            P = pooled[e].reshape(B * T, -1)
            if T % 64 == 0:
                # ONE pass per encoder: with G_b = dOut[b]^T P_e[b] (the accumulator, drained once per video), dW_e = sum_b w_e[b] G_b and
                # <Z_e[b], P_e[b]> = <W_e, G_b> — the Z_e = dOut W_e GEMM and the pair-dot pass below are not needed (half the tensor work)
                dW, dwp = ops.wgrad_video(g, P, weights[:, e], Ws[e], B)
                dw_partials.append(dwp)
                pbars.append(ops.video_colsum(P.reshape(B, T, -1), 1.0 / T))
                dWs.append(dW)
                continue
            Z = ops.gemm_ex(g, Ws[e], w_t=True)  # dOut W_e : [M, K] x [K, C_e] -> [M, C_e]
            dwp, Ps = ops.pair_dot(Z.reshape(B, -1), P.reshape(B, -1), scale=weights[:, e])  # <Z_e, P_e> partials and w_e (.) P_e in one pass
            dw_partials.append(dwp)
            pbars.append(ops.video_colsum(P.reshape(B, T, -1), 1.0 / T))
            dWs.append(ops.gemm_ex(g, Ps.view(B * T, -1), a_t=True, w_t=True))  # dOut^T (w_e (.) P_e) : contraction over the tokens -> [K, C_e]
        _, dbs, dQ, dWq, dWk, dbias = ops.fused_backward(weights, dwo, u, gsum, dw_partials, pbars, Ws, biases, Qc, Wqc, Wkc, bc, dWs)
        grads = [dQ.reshape(1, -1), dWq, dWk, dbias]
        for e in range(E):
            grads += [dWs[e], dbs[e]]
        grads = [gr.to(pd) if gr is not None else None for gr, pd in zip(grads, ctx.param_dtypes)]
        return (None, None, None, None, None, demb, *grads)


class _FusedScalarLinearFn(torch.autograd.Function):
    """Training step of 3d-avg / avg pool + linear projectors + ScalarAdapter through the fused forward (pool -> softmax(scalar) ->
    merv_fused_linear_mix), with a backward that never materialises the per-encoder projections Y_e or their gradients dV_e.

    backward: per encoder ONE tcgen05 pass over dOut and the pooled tokens P_e (merv_wgrad_video, the same w_e for every video):
              dW_e = w_e dOut^T P_e and the partials of <dOut[b], Y_e[b] - b_e>;  gsum = colsum_t(dOut);  then merv_scalar_fused_backward:
              db_e = w_e sum_b gsum[b],  g_e = partials + b_e . sum_b gsum[b] + dW_out[e],  dscalar = w (.) (g - <w, g>).
    Needs T % 64 == 0 (ScalarAdapter._can_fuse_training); no gradient flows into the patch features (frozen backbones).  ``batch_index`` and
    an assembly (``asm``) as for _FusedLinearFn."""

    @staticmethod
    def forward(ctx, adapter, projs, xs, batch_index, asm, emb, scalar, *proj_params):
        dtype = torch.bfloat16
        E, B = len(projs), (xs[0].shape[0] if batch_index is None else batch_index.numel())
        lasts = [p.layers()[0][0] for p in projs]
        Ws = [p._cast_cache.get(lin.weight, dtype) for lin, p in zip(lasts, projs)]
        biases = [p._cast_cache.get(lin.bias, dtype) for lin, p in zip(lasts, projs)]
        pooled, _ = ops.pool3d(xs, [p.output_frames for p in projs], projs[0].output_size, batch_index=batch_index)
        T, K = pooled[0].shape[1], lasts[0].out_features
        scores = scalar.detach().float().reshape(1, E).expand(B, E).contiguous()
        weights, bias_mix = ops.softmax_weights(scores, biases, K)
        out, buf = _fused_mix_into(asm, pooled, Ws, weights, bias_mix, B, T, K)
        ctx.dims = (B, E, T, K)
        ctx.asm = asm
        ctx.param_dtypes = [t.dtype for t in (scalar, *proj_params)]
        ctx.save_for_backward(weights[0], *pooled, *Ws, *biases)
        return (out if asm is None else buf), weights[:1].to(dtype)

    @staticmethod
    def backward(ctx, dout, dweights):
        B, E, T, K = ctx.dims
        w, *saved = ctx.saved_tensors
        pooled, Ws, biases = saved[:E], saved[E:2 * E], saved[2 * E:3 * E]
        dt = Ws[0].dtype
        g, demb = _fused_dout(ctx.asm, dout, B, T, K, dt, w.device, ctx.needs_input_grad[5])
        gsum = ops.video_colsum(g.view(B, T, K))
        dWs, dw_partials = [], []
        for e in range(E):  # scale stride 0: w_e for every video
            dW, dwp = ops.wgrad_video(g, pooled[e].reshape(B * T, -1), w[e].expand(B), Ws[e], B)
            dWs.append(dW)
            dw_partials.append(dwp)
        dwo = None if dweights is None else dweights.float().reshape(-1).contiguous()
        dscalar, dbs = ops.scalar_fused_backward(w, dwo, gsum, dw_partials, biases)
        grads = [dscalar]
        for e in range(E):
            grads += [dWs[e], dbs[e]]
        grads = [gr.to(pd) if gr is not None else None for gr, pd in zip(grads, ctx.param_dtypes)]
        return (None, None, None, None, None, demb, *grads)


def _unwrap(module: nn.Module) -> nn.Module:
    """The module behind an FSDP1 wrapper (FSDP(LinearProjector) is what the reference's wrap policy, merv.py:473-485, turns the
    inner ``projector`` of every resampler into); anything else is returned unchanged."""
    return getattr(module, "_fsdp_wrapped_module", module)


def _projector_layers(projector: nn.Module) -> List[Tuple[nn.Linear, int]]:
    """[(linear, activation applied AFTER it)] for every reference projector type."""
    projector = _unwrap(projector)
    if isinstance(projector, LinearProjector):
        return [(projector.projector, ACT_NONE)]
    if isinstance(projector, (MLPProjector, MLPDeepProjector, FusedMLPProjector)):
        mods = list(projector.projector)
        layers = []
        for i, m in enumerate(mods):
            if isinstance(m, nn.Linear):
                act = ACT_GELU_ERF if i + 1 < len(mods) and isinstance(mods[i + 1], nn.GELU) else ACT_NONE
                layers.append((m, act))
        return layers
    if isinstance(projector, nn.Identity):
        return []
    raise TypeError(f"unsupported projector module {type(projector).__name__}")


def _run_layers(x: torch.Tensor, layers, cache: _CastCache, dtype: torch.dtype, last_rowdot_vec=None, train: bool = False,
                ln: Optional[nn.LayerNorm] = None):
    rd = None
    if train:
        if any(lin.bias is None for lin, _ in layers) or (ln is not None and (ln.weight is None or ln.bias is None)):
            raise NotImplementedError("bias-free projector layers / non-affine LayerNorm are not covered by the backward")
        params = ([ln.weight, ln.bias] if ln is not None else []) + [t for lin, _ in layers for t in (lin.weight, lin.bias)]
        return _ProjectorFn.apply(x, tuple(act for _, act in layers), dtype, cache, None if ln is None else ln.eps, *params), None
    if ln is not None:
        x = ops.layernorm([x], cache.get(ln.weight, dtype), cache.get(ln.bias, dtype), ln.eps)
    for i, (lin, act) in enumerate(layers):
        rv = last_rowdot_vec if i == len(layers) - 1 else None
        x, rd = ops.linear_bias_act(x, cache.get(lin.weight, dtype), cache.get(lin.bias, dtype), act, rv)
    return x, rd


# === Definitions for Various Projection Modules, with Signature :: [..., in_dim] --> [..., out_dim] ===
class _ProjectorBase(nn.Module):
    def _pre_ln(self) -> Optional[nn.LayerNorm]:
        """The nn.LayerNorm of `pre_proj_layernorm=True` (nn_utils.py:26-29), None for the nn.Identity default."""
        ln = self.layernorm
        if isinstance(ln, nn.Identity):
            return None
        if not isinstance(ln, nn.LayerNorm) or len(ln.normalized_shape) != 1:
            raise TypeError(f"unsupported pre-projection normalisation {type(ln).__name__}")
        return ln

    def forward(self, img_patches: torch.Tensor) -> torch.Tensor:
        _require_device(img_patches)
        ln = self._pre_ln()
        train = _needs_grad(self, img_patches)
        dtype = _compute_dtype(img_patches)
        if not hasattr(self, "_cast_cache"):
            self._cast_cache = _CastCache()
        x = img_patches if img_patches.dtype == dtype else img_patches.to(dtype)
        layers = _projector_layers(self)
        if x.numel() == 0:
            return torch.empty((*x.shape[:-1], layers[-1][0].out_features), dtype=dtype, device=x.device)
        y, _ = _run_layers(x, layers, self._cast_cache, dtype, train=train, ln=ln)
        return y


class LinearProjector(_ProjectorBase):
    def __init__(self, vision_dim: int, llm_dim: int, pre_proj_layernorm: bool = False) -> None:
        super().__init__()
        self.projector = nn.Linear(vision_dim, llm_dim, bias=True)
        if pre_proj_layernorm:
            self.layernorm = nn.LayerNorm(vision_dim)
        else:
            self.layernorm = nn.Identity()


class MLPProjector(_ProjectorBase):
    def __init__(
        self, vision_dim: int, llm_dim: int, mlp_type: str = "gelu-mlp", pre_proj_layernorm: bool = False
    ) -> None:
        super().__init__()
        if pre_proj_layernorm:
            self.layernorm = nn.LayerNorm(vision_dim)
        else:
            self.layernorm = nn.Identity()
        if mlp_type == "gelu-mlp":
            self.projector = nn.Sequential(
                nn.Linear(vision_dim, llm_dim, bias=True),
                nn.GELU(),
                nn.Linear(llm_dim, llm_dim, bias=True),
            )
        else:
            raise ValueError(f"Projector with `{mlp_type = }` is not supported!")

    @property
    def output_token_length(self) -> int:
        return 1


class MLPDeepProjector(_ProjectorBase):
    def __init__(
        self, vision_dim: int, llm_dim: int, mlp_type: str = "gelu-mlp", pre_proj_layernorm: bool = False
    ) -> None:
        super().__init__()
        if pre_proj_layernorm:
            self.layernorm = nn.LayerNorm(vision_dim)
        else:
            self.layernorm = nn.Identity()
        if mlp_type == "gelu-mlp":
            self.projector = nn.Sequential(
                nn.Linear(vision_dim, llm_dim, bias=True),
                nn.GELU(),
                nn.Linear(llm_dim, llm_dim, bias=True),
                nn.GELU(),
                nn.Linear(llm_dim, llm_dim, bias=True),
            )
        else:
            raise ValueError(f"Projector with `{mlp_type = }` is not supported!")


class FusedMLPProjector(_ProjectorBase):
    def __init__(
        self, fused_vision_dim: int, llm_dim: int, mlp_type: str = "fused-gelu-mlp", pre_proj_layernorm: bool = False
    ) -> None:
        super().__init__()
        if pre_proj_layernorm:
            self.layernorm = nn.LayerNorm(fused_vision_dim)
        else:
            self.layernorm = nn.Identity()
        self.initial_projection_dim = fused_vision_dim * 4
        if mlp_type == "fused-gelu-mlp":
            self.projector = nn.Sequential(
                nn.Linear(fused_vision_dim, self.initial_projection_dim, bias=True),
                nn.GELU(),
                nn.Linear(self.initial_projection_dim, llm_dim, bias=True),
                nn.GELU(),
                nn.Linear(llm_dim, llm_dim, bias=True),
            )
        else:
            raise ValueError(f"Fused Projector with `{mlp_type = }` is not supported!")


def get_mlp_projector(fused_vision_dim: int, llm_dim: int, mlp_type: str = "gelu-mlp") -> nn.Module:
    if mlp_type == "linear":
        return LinearProjector(fused_vision_dim, llm_dim)
    elif mlp_type == "gelu-mlp":
        return MLPProjector(fused_vision_dim, llm_dim, mlp_type)
    elif mlp_type == "fused-gelu-mlp":
        return FusedMLPProjector(fused_vision_dim, llm_dim, mlp_type)
    elif mlp_type == "none":
        return nn.Identity()
    else:
        raise ValueError(f"Projector with `{mlp_type = }` is not supported!")


class TokenResampler(nn.Module, ABC):
    """Resamples token length as well. Abstract class for interfacing resulting token length."""

    @property
    @abstractmethod
    def output_token_length(self) -> int: ...

    @property
    @abstractmethod
    def output_frame_length(self) -> int: ...


class DeferredProjection:
    """What a *linked* ``AveragePooling3DProjector`` returns: the un-projected features plus the module that owns
    the weights.  ``MERV.forward`` only threads the projector outputs into ``feature_fusion`` (merv.py:587-589,608),
    which consumes these and runs the fused pipeline.  ``materialize()`` gives the ordinary tensor."""

    def __init__(self, projector: "AveragePooling3DProjector", features: torch.Tensor) -> None:
        self.projector, self.features = projector, features

    @property
    def shape(self) -> torch.Size:
        p = self.projector
        return torch.Size((self.features.shape[0], p.output_frames * p.output_size * p.output_size, p.llm_dim))

    @property
    def dtype(self) -> torch.dtype:
        return _compute_dtype(self.features)

    @property
    def device(self) -> torch.device:
        return self.features.device

    def materialize(self) -> torch.Tensor:
        return self.projector._forward_unfused(self.features)


def _materialize(V, batch_index: Optional[torch.Tensor]) -> List[torch.Tensor]:
    """Projected tokens of the videos `batch_index` selects (all when None).  A DeferredProjection still holds the whole batch's features:
    they are gathered with index_select before the projector runs, as the reference indexes the inputs before the backbones (merv.py:576-585);
    tensors are the outputs of projectors that already saw the gathered features (MervFusion._project)."""
    out = []
    for v in V:
        if isinstance(v, DeferredProjection):
            x = v.features if batch_index is None else v.features.index_select(0, batch_index.to(device=v.features.device, dtype=torch.long))
            v = v.projector._forward_unfused(x)
        out.append(v)
    return out


class AveragePooling3DProjector(TokenResampler):
    """3D-average pooling projector (pool FIRST, then project: nn_utils.py:328-330)."""

    def __init__(
        self, fused_vision_dim: int, llm_dim: int, output_frames: int, output_size: int, mlp_type: str = "gelu-mlp"
    ) -> None:
        super().__init__()
        self.output_frames = output_frames
        self.output_size = output_size
        self.llm_dim = llm_dim
        self.fused_vision_dim = fused_vision_dim
        # kept for state-dict/module-tree parity with the reference (it has no parameters)
        self.avg_pooling = nn.AdaptiveAvgPool3d((output_frames, output_size, output_size))
        self.projector = get_mlp_projector(fused_vision_dim, llm_dim, mlp_type)
        self._cast_cache = _CastCache()
        self._linked_fusion = None  # weakref to the adapter when linked

    @classmethod
    def from_reference(cls, ref_module: nn.Module) -> "AveragePooling3DProjector":
        """Adopt a reference ``AveragePooling3DProjector``: same ``projector`` submodule objects (parameters shared)."""
        inner = ref_module.projector
        lins = [m for m in inner.modules() if isinstance(m, nn.Linear)]
        if not lins:
            raise ValueError("reference projector has no Linear layer (mlp_type 'none' has nothing to accelerate)")
        n = len(lins)
        mlp_type = {1: "linear", 2: "gelu-mlp", 3: "fused-gelu-mlp"}[n]
        new = cls(lins[0].in_features, lins[-1].out_features, ref_module.output_frames, ref_module.output_size, mlp_type)
        new.projector.projector = inner.projector  # nn.Linear ("linear") or the nn.Sequential of the MLP types: shared, not copied
        return new

    def layers(self) -> List[Tuple[nn.Linear, int]]:
        return _projector_layers(self.projector)

    def _forward_unfused(self, fused_img_patches: torch.Tensor):
        """pool -> ``self.projector(pooled)``.  The inner projector is CALLED as a module, exactly as the reference does
        (nn_utils.py:330): under the reference's FSDP policy it is its own unit (merv.py:473-485) and its parameters only exist
        unsharded inside its own forward."""
        dtype = _compute_dtype(fused_img_patches)
        if torch.is_grad_enabled() and fused_img_patches.requires_grad:
            raise NotImplementedError("gradients w.r.t. the patch features are not implemented (frozen backbones, merv.py:316)")
        x = fused_img_patches.detach()
        x = x if x.dtype == dtype else x.to(dtype)
        if x.shape[0] == 0:
            return torch.empty((0, self.output_frames * self.output_size**2, self.llm_dim), dtype=dtype, device=x.device)
        (pooled,), _ = ops.pool3d([x], [self.output_frames], self.output_size)
        return self.projector(pooled)

    def forward(self, fused_img_patches: torch.Tensor) -> Union[torch.Tensor, DeferredProjection]:
        assert fused_img_patches.dim() == 4, "expected [B, F, N, C] patch features (merv.py:576-585)"
        _require_device(fused_img_patches)
        fusion = self._linked_fusion() if self._linked_fusion is not None else None
        if fusion is not None:
            # Deferring moves the read of THIS module's weights into the adapter's forward.  Under FSDP with per-projector units
            # (merv.py:473-485) they are resharded again by then — in eval / no_grad passes just as in training.
            defer = fusion._may_defer(self) if hasattr(fusion, "_may_defer") else not torch.is_grad_enabled()
            if defer:
                return DeferredProjection(self, fused_img_patches)
        return self._forward_unfused(fused_img_patches)

    @property
    def output_token_length(self) -> int:
        return self.output_size * self.output_size

    @property
    def output_frame_length(self) -> int:
        return self.output_frames


class AveragePoolingProjector(AveragePooling3DProjector):
    """Emu-2 style projector: n x n average pooling of every frame, then the projector (nn_utils.py:136-174).

    Same kernels as the 3-D resampler with an identity temporal window (the reference asserts num_frames ==
    output_frames, nn_utils.py:155); state-dict keys and constructor signature are the reference's (note the argument
    order: output_size before output_frames, and the ``avg_pool`` attribute name)."""

    def __init__(
        self, fused_vision_dim: int, llm_dim: int, output_size: int, output_frames: int = 8, mlp_type: str = "gelu-mlp"
    ) -> None:
        super().__init__(fused_vision_dim, llm_dim, output_frames, output_size, mlp_type)
        del self.avg_pooling
        self.avg_pool = nn.AdaptiveAvgPool2d((output_size, output_size))

    @classmethod
    def from_reference(cls, ref_module: nn.Module) -> "AveragePoolingProjector":
        lins = [m for m in ref_module.projector.modules() if isinstance(m, nn.Linear)]
        if not lins:
            raise ValueError("reference projector has no Linear layer (mlp_type 'none' has nothing to accelerate)")
        mlp_type = {1: "linear", 2: "gelu-mlp", 3: "fused-gelu-mlp"}[len(lins)]
        new = cls(lins[0].in_features, lins[-1].out_features, ref_module.output_size, ref_module.output_frames, mlp_type)
        new.projector.projector = ref_module.projector.projector
        return new

    def forward(self, fused_img_patches: torch.Tensor):
        assert fused_img_patches.dim() == 4
        assert fused_img_patches.shape[1] == self.output_frames  # nn_utils.py:154-155
        return super().forward(fused_img_patches)


class Convolutional3DProjector(TokenResampler):
    """3D-convolutional projector ("3dconv" resampler, nn_utils.py:341-377; constructed at merv.py:142-150): Conv3d(C -> llm_dim, 3 x 3 x 3,
    padding 1) -> AdaptiveAvgPool3d -> projector(llm_dim -> llm_dim).

    B200 form: the pool is linear and the convolution is a sum over 27 displaced copies of the input, so
    ``pool(conv(x)) = sum_tap W_tap pool(shift_tap(x)) + b``: the pool kernel writes the 27 displaced poolings side by side (5-D TMA loads
    with displaced box coordinates; the TMA unit zero-fills what falls outside the grid = the convolution's zero padding) and ONE tcgen05
    GEMM with K = 27 C evaluates the convolution on the POOLED grid — T*S*S instead of F*H*W positions per video, no channel-major
    permute, no im2col of the un-pooled features.  Module tree, parameter names and init order are the reference's."""

    def __init__(
        self, fused_vision_dim: int, llm_dim: int, output_frames: int, output_size: int, mlp_type: str = "gelu-mlp"
    ) -> None:
        super().__init__()
        self.output_frames = output_frames
        self.output_size = output_size
        self.convolution_pooling = nn.Sequential(
            nn.Conv3d(fused_vision_dim, llm_dim, kernel_size=3, stride=1, padding=1),
            nn.AdaptiveAvgPool3d((output_frames, output_size, output_size)),
        )
        self.projector = get_mlp_projector(llm_dim, llm_dim, mlp_type)
        self._conv_cache = None

    @classmethod
    def from_reference(cls, ref_module: nn.Module) -> "Convolutional3DProjector":
        """Adopt a reference ``Convolutional3DProjector``: the Conv3d and the inner projector are shared, not copied."""
        conv = ref_module.convolution_pooling[0]
        assert isinstance(conv, nn.Conv3d) and conv.kernel_size == (3, 3, 3) and conv.stride == (1, 1, 1) and conv.padding == (1, 1, 1) \
            and conv.dilation == (1, 1, 1) and conv.groups == 1 and conv.padding_mode == "zeros"
        new = cls.__new__(cls)
        nn.Module.__init__(new)
        new.output_frames, new.output_size = ref_module.output_frames, ref_module.output_size
        new.convolution_pooling = ref_module.convolution_pooling
        new.projector = _adopt_plain_projector(ref_module.projector) if type(ref_module.projector).__name__ in _PLAIN_PROJECTORS else ref_module.projector
        new._conv_cache = None
        return new

    def _conv_operands(self, dtype: torch.dtype):
        """(W2 [K, 27 C] tap-major — column (kf*9 + kh*3 + kw) * C + c holds weight[k, c, kf, kh, kw] — and the bias), in the compute dtype;
        rebuilt when the parameters change (version counter) and never cached for FSDP views."""
        conv = _unwrap(self.convolution_pooling[0])
        w, b = conv.weight, conv.bias
        tag = (w.data_ptr(), _version(w), None if b is None else (b.data_ptr(), _version(b)), dtype)
        hit = self._conv_cache
        if hit is not None and hit[0] == tag and not (_is_volatile(w) or _is_volatile(b)):
            return hit[1], hit[2]
        with torch.no_grad():
            W2 = w.detach().to(dtype).permute(0, 2, 3, 4, 1).reshape(w.shape[0], -1).contiguous()
            b2 = None if b is None else b.detach().to(dtype).contiguous()
        self._conv_cache = (tag, W2, b2)
        return W2, b2

    def forward(self, fused_img_patches: torch.Tensor) -> torch.Tensor:
        assert fused_img_patches.dim() == 4  # nn_utils.py:361
        _require_device(fused_img_patches)
        dtype = _compute_dtype(fused_img_patches)
        if torch.is_grad_enabled() and fused_img_patches.requires_grad:
            raise NotImplementedError("gradients w.r.t. the patch features are not implemented (frozen backbones, merv.py:316)")
        x = fused_img_patches.detach()
        x = x if x.dtype == dtype else x.to(dtype)
        if not _tma_readable(x):
            x = x.contiguous()
        conv = _unwrap(self.convolution_pooling[0])
        if x.shape[0] == 0:
            return self.projector(torch.empty((0, self.output_frames * self.output_size**2, conv.out_channels), dtype=dtype, device=x.device))
        A = ops.pool3d_conv_taps(x, self.output_frames, self.output_size)
        if _needs_grad(conv):
            y = _ConvTapsFn.apply(A, dtype, self, conv.weight, conv.bias)
        else:
            W2, b = self._conv_operands(dtype)
            y, _ = ops.linear_bias_act(A, W2, b, ACT_NONE)
        return self.projector(y.reshape(A.shape[0], A.shape[1], -1))

    @property
    def output_token_length(self) -> int:
        return self.output_size * self.output_size

    @property
    def output_frame_length(self) -> int:
        return self.output_frames


class CrossAttention(nn.Module):
    """Parameter container with the reference's attribute names (merv/util/nn_utils.py:380-391); the arithmetic of its forward
    (:393-412) runs in AttentivePooler.forward below."""

    def __init__(self, dim, num_heads=12, qkv_bias=False, use_sdpa=True):
        super().__init__()
        self.num_heads = num_heads
        head_dim = dim // num_heads
        self.scale = head_dim**-0.5
        self.q = nn.Linear(dim, dim, bias=qkv_bias)
        self.kv = nn.Linear(dim, int(dim * 2), bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)
        self.use_sdpa = use_sdpa


class MLP(nn.Module):
    """merv/util/nn_utils.py:415-423 (parameter container)."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.0):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)


class CrossAttentionBlock(nn.Module):
    """merv/util/nn_utils.py:434-445 (parameter container)."""

    def __init__(self, dim, num_heads, mlp_ratio=4.0, qkv_bias=False, out_dim=None, act_layer=nn.GELU, norm_layer=nn.LayerNorm):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.xattn = CrossAttention(dim, num_heads=num_heads, qkv_bias=qkv_bias)
        self.norm2 = norm_layer(dim)
        mlp_hidden_dim = int(dim * mlp_ratio)
        self.mlp = MLP(in_features=dim, hidden_features=mlp_hidden_dim, out_features=out_dim, act_layer=act_layer)


class AttentivePooler(TokenResampler):
    """Attentive pooler from JEPA, the "attntv" resampler (merv/util/nn_utils.py:177-246; merv.py:124-130): every frame's N patch tokens
    are resampled to ``num_query_tokens`` tokens by one cross-attention block with learned queries, then projected.

    Same constructor signature, module tree (hence state-dict keys: ``query_tokens``, ``cross_attn.{norm1,xattn.{q,kv,proj},norm2,
    mlp.{fc1,fc2}}``, ``projector.*``) and initialisation sequence as the reference.  forward: LayerNorm (merv_layernorm), the kv / proj /
    MLP / projector Linears on the tcgen05 GEMM (GELU in the epilogue), merv_cross_attention (both contractions as tcgen05.mma in bf16),
    merv_add_rows for the two residuals.  Training, in fp32 or bf16 compute, wherever the forward runs: _AttentivePoolFn, a hand-written
    backward whose attention part is merv_cross_attention_backward_ex (five tcgen05 contractions per frame and head for bf16 frames of
    at most 64 queries and 256 keys with head_dim % 32 == 0, the CUDA-core kernel otherwise)."""

    def __init__(self, fused_vision_dim: int, llm_dim: int, num_query_tokens: int, num_heads: int = 8, output_frames: int = 8,
                 mlp_type: str = "gelu-mlp") -> None:
        super().__init__()
        self.num_query_tokens = num_query_tokens
        self.output_frames = output_frames
        assert fused_vision_dim % num_heads == 0, "fused_vision_dim must be divisible by num_heads"

        self.query_tokens = nn.Parameter(torch.zeros(1, num_query_tokens, fused_vision_dim))
        self.cross_attn = CrossAttentionBlock(dim=fused_vision_dim, num_heads=num_heads, qkv_bias=True)
        self.projector = get_mlp_projector(fused_vision_dim, llm_dim, mlp_type)

        nn.init.trunc_normal_(self.query_tokens, std=0.02)
        self.apply(self._init_weights)
        self._rescale_blocks()
        self._cast_cache = _CastCache()

    def _rescale_blocks(self):
        def rescale(param, layer_id):
            param.div_(math.sqrt(2.0 * layer_id))

        rescale(self.cross_attn.xattn.proj.weight.data, 1)
        rescale(self.cross_attn.mlp.fc2.weight.data, 1)

    def _init_weights(self, m):
        init_std = 0.02
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=init_std)
            if isinstance(m, nn.Linear) and m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)

    @classmethod
    def from_reference(cls, ref_module: nn.Module) -> "AttentivePooler":
        """Adopt a reference ``AttentivePooler``: its ``query_tokens``, ``cross_attn`` and projector sub-modules are shared, not copied."""
        new = cls.__new__(cls)
        nn.Module.__init__(new)
        new.num_query_tokens, new.output_frames = ref_module.num_query_tokens, ref_module.output_frames
        new.query_tokens, new.cross_attn = ref_module.query_tokens, ref_module.cross_attn
        new.projector = _adopt_plain_projector(ref_module.projector)
        new._cast_cache = _CastCache()
        return new

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        # x: [B, F, N, C]
        assert x.dim() == 4, "expected [B, F, N, C] patch features (merv.py:576-585)"
        num_frames = x.shape[1]
        assert num_frames == self.output_frames  # nn_utils.py:232
        _require_device(x)
        dtype = _compute_dtype(x)
        c = self._cast_cache
        blk, att = self.cross_attn, self.cross_attn.xattn
        B, F, N, C_ = x.shape
        n = self.num_query_tokens
        layers = _projector_layers(self.projector)
        if B == 0:
            return torch.empty((0, F * n, layers[-1][0].out_features), dtype=dtype, device=x.device)
        if _needs_grad(self, x):
            if x.requires_grad:
                raise NotImplementedError("gradients w.r.t. the patch features are not implemented (frozen backbones, merv.py:316)")
            lins = (att.kv, att.q, att.proj, blk.mlp.fc1, blk.mlp.fc2)
            if any(l.bias is None for l in lins) or any(ln.weight is None or ln.bias is None for ln in (blk.norm1, blk.norm2)):
                raise NotImplementedError("bias-free layers / non-affine LayerNorms of the attentive pooler are not covered by the backward")
            xb = x.detach()
            xb = xb if xb.dtype == dtype else xb.to(dtype)
            q2 = _AttentivePoolFn.apply(xb, dtype, c, att.num_heads, att.scale, blk.norm1.eps, blk.norm2.eps, self.query_tokens, blk.norm1.weight,
                                        blk.norm1.bias, att.kv.weight, att.kv.bias, att.q.weight, att.q.bias, att.proj.weight, att.proj.bias,
                                        blk.norm2.weight, blk.norm2.bias, blk.mlp.fc1.weight, blk.mlp.fc1.bias, blk.mlp.fc2.weight, blk.mlp.fc2.bias)
            out = self.projector(q2)
            return out.view(B, F * n, out.shape[-1])
        xf = (x if x.dtype == dtype else x.to(dtype)).reshape(B * F * N, C_)
        xn = ops.layernorm([xf], c.get(blk.norm1.weight, dtype), c.get(blk.norm1.bias, dtype), blk.norm1.eps)
        kv, _ = ops.linear_bias_act(xn, c.get(att.kv.weight, dtype), c.get(att.kv.bias, dtype), ACT_NONE)  # [B F N, 2C] = [K | V]
        qt = c.get(self.query_tokens, dtype)[0]  # the same learned queries for every frame (nn_utils.py:234)
        qp, _ = ops.linear_bias_act(qt, c.get(att.q.weight, dtype), c.get(att.q.bias, dtype), ACT_NONE)
        a = ops.cross_attention(qp, kv, B * F, att.num_heads, att.scale)  # [B F, n, C]
        y, _ = ops.linear_bias_act(a.view(B * F * n, C_), c.get(att.proj.weight, dtype), c.get(att.proj.bias, dtype), ACT_NONE)
        q1 = ops.add_rows(y, qt)  # q + xattn(q, norm1(x)), q = the query tokens of every frame
        h = ops.layernorm([q1], c.get(blk.norm2.weight, dtype), c.get(blk.norm2.bias, dtype), blk.norm2.eps)
        h, _ = ops.linear_bias_act(h, c.get(blk.mlp.fc1.weight, dtype), c.get(blk.mlp.fc1.bias, dtype), ACT_GELU_ERF)
        h, _ = ops.linear_bias_act(h, c.get(blk.mlp.fc2.weight, dtype), c.get(blk.mlp.fc2.bias, dtype), ACT_NONE)
        q2 = ops.add_rows(q1, h)  # q + mlp(norm2(q))
        out = self.projector(q2)  # called as a module: its own FSDP unit under the reference's policy (merv.py:473-485)
        return out.view(B, F * n, out.shape[-1])  # "(B F) N C -> B (F N) C"

    @property
    def output_token_length(self) -> int:
        return self.num_query_tokens

    @property
    def output_frame_length(self) -> int:
        return self.output_frames


# Adapters here
class _LinkedMixer(nn.Module):
    """When linked projectors hand their input over to a mixer (DeferredProjection) instead of projecting it themselves.  Shared by the
    mixers that run a fused path: CrossAttentionAdapterLearnableQuery and ScalarAdapter."""

    # True / False force the training step onto / off the fused path (_FusedLinearFn, _FusedScalarLinearFn); None (default) decides per
    # call: fused unless a parameter involved is managed by FSDP.  The fused path reads every projector's parameters inside the mixer's
    # forward, and per-projector FSDP units (merv.py:473-485) have resharded them by then; wrap MervFusion as one unit (INTEGRATION.md)
    # and set True to use it under FSDP.
    fused_training: Optional[bool] = None

    def _defer_in_grad_mode(self, projector: nn.Module) -> bool:
        """Whether a linked projector should hand its input over (DeferredProjection) although autograd is recording."""
        if self.fused_training is not None:
            return bool(self.fused_training)
        return not any(_is_sharded_param(p) for m in (self, projector) for p in m.parameters())

    def _may_defer(self, projector: nn.Module) -> bool:
        """Whether a linked projector hands its input over to this mixer instead of projecting it itself.  The fused pipeline
        reads the projector's weights inside THIS module's forward, so parameters managed by a different FSDP unit (already
        resharded by then) rule it out — with or without autograd — unless ``fused_training=True`` states that projectors and
        mixer share one unit."""
        if torch.is_grad_enabled():
            return self._defer_in_grad_mode(projector)
        if self.fused_training:
            return True
        return not any(_is_sharded_param(p) for m in (self, projector) for p in m.parameters())


class CrossAttentionAdapterLearnableQuery(_LinkedMixer):
    def __init__(
        self, embed_dim=3072, llm_dim=4098, token_length=8, averagetoken=False, num_encoder=4, positional_embedding=False
    ) -> None:
        super().__init__()
        self.llm_dim = llm_dim
        self.token_length = token_length
        self.averagetoken = averagetoken
        # parameter container only: forward never calls it (v_proj_weight / out_proj are dead in the reference too)
        self.attention = nn.MultiheadAttention(
            embed_dim=embed_dim,
            num_heads=1,
            dropout=0.0,
            batch_first=True,
            kdim=llm_dim if averagetoken else token_length * llm_dim,
            vdim=llm_dim if averagetoken else token_length * llm_dim,
        )
        self.Q = Parameter(torch.empty((1, embed_dim)))
        self.num_encoder = num_encoder
        self.positional_embedding = positional_embedding
        if positional_embedding:
            self.pe = Parameter(torch.empty((self.num_encoder, llm_dim)))
        self._reset_parameters()
        self._cast_cache = _CastCache()
        self._u_cache = {}
        self._vc_cache = {}
        self.fused_training: Optional[bool] = None  # see _LinkedMixer

    def _reset_parameters(self):
        xavier_uniform_(self.Q)
        if self.positional_embedding:
            xavier_uniform_(self.pe)

    @classmethod
    def from_reference(cls, ref_module: nn.Module) -> "CrossAttentionAdapterLearnableQuery":
        att = ref_module.attention
        new = cls(att.embed_dim, ref_module.llm_dim, ref_module.token_length, ref_module.averagetoken,
                  ref_module.num_encoder, ref_module.positional_embedding)
        new.attention, new.Q = att, ref_module.Q
        if ref_module.positional_embedding:
            new.pe = ref_module.pe
        return new

    # ---- cached, input-independent vectors ----------------------------------------------------------------
    def query_vector(self, dtype: torch.dtype) -> torch.Tensor:
        """u (fp32 [llm_dim]) with weights == softmax_e(u . mean_t V_e); recomputed when a parameter changes."""
        att = self.attention
        params = (self.Q, att.q_proj_weight, att.k_proj_weight, att.in_proj_bias)
        tag = tuple((p.data_ptr(), _version(p)) for p in params if p is not None) + (dtype, self.Q.device)
        hit = self._u_cache.get("u")
        if hit is None or hit[0] != tag or any(_is_volatile(p) for p in params):
            c = self._cast_cache
            u = ops.fusion_query_vec(c.get(self.Q, dtype), c.get(att.q_proj_weight, dtype), c.get(att.k_proj_weight, dtype),
                                     c.get(att.in_proj_bias, dtype))
            hit = (tag, u)
            self._u_cache["u"] = hit
            self._vc_cache.clear()
        return hit[1]

    def _affine_vec(self, lin: nn.Linear, cache: _CastCache, dtype: torch.dtype):
        """(v, c) for the last (affine) projector layer: u . (W x + b) = v . x + c."""
        u = self.query_vector(dtype)
        tag = (lin.weight.data_ptr(), _version(lin.weight), None if lin.bias is None else _version(lin.bias), dtype, id(u))
        hit = self._vc_cache.get(id(lin))
        if hit is None or hit[0] != tag or _is_volatile(lin.weight) or _is_volatile(lin.bias):
            hit = (tag, ops.affine_score_vec(cache.get(lin.weight, dtype), cache.get(lin.bias, dtype), u))
            self._vc_cache[id(lin)] = hit
        return hit[1]

    def _pe_consts(self, dtype: torch.dtype, c_in=None) -> Optional[torch.Tensor]:
        """fp32 [E] with c[e] = u . pe[e] (+ c_in[e]): positional_embedding=True adds pe[e] to encoder e's mean token before
        the attention (nn_utils.py:510-511), i.e. a constant to its score.  None when the module has no ``pe`` or runs with
        averagetoken=False (the reference only uses ``pe`` inside the averagetoken branch)."""
        if not (self.positional_embedding and self.averagetoken):
            return None
        u = self.query_vector(dtype)
        tag = (self.pe.data_ptr(), _version(self.pe), id(u), None if c_in is None else tuple(id(c) for c in c_in))
        hit = self._u_cache.get("pe")
        if hit is None or hit[0] != tag or _is_volatile(self.pe):
            hit = (tag, ops.score_consts(self._cast_cache.get(self.pe, dtype), u, c_in), c_in)  # c_in kept alive: ids are the key
            self._u_cache["pe"] = hit
        return hit[1]

    # ---- forward --------------------------------------------------------------------------------------------
    def forward(self, V, out: Optional[torch.Tensor] = None, batch_index: Optional[torch.Tensor] = None, gather=None):
        # V is a list of tensors with size (B, T, K). T should all be same, or 1.  (nn_utils.py:491-495)
        # `out` / `batch_index` are extensions of the linked (fused) path only, see _forward_fused.
        for emb in V:
            assert emb.shape[1] == self.token_length or emb.shape[1] == 1, (self.token_length, [e.shape for e in V])
        assert 1 <= len(V) <= 8, f"1..8 encoders supported, got {len(V)}"
        if self.positional_embedding and self.averagetoken:
            assert len(V) == self.num_encoder, f"pe holds {self.num_encoder} rows, got {len(V)} encoders (nn_utils.py:511)"
        if V[0].shape[0] == 0:  # a rank that owns no videos (merv_b200/parallel.py): nothing to launch
            dt, dev = (V[0].dtype, V[0].device)
            return torch.empty((0, self.token_length, self.llm_dim), dtype=dt, device=dev), torch.empty((0, len(V)), dtype=dt, device=dev)

        deferred = all(isinstance(v, DeferredProjection) for v in V)
        if deferred and torch.is_grad_enabled() and _needs_grad(self, *[t for v in V for t in v.projector.parameters()]):
            if out is None and batch_index is None and gather is None and self._can_fuse_training(V):
                return self._forward_fused_train(V)
        elif deferred and self._can_fuse(V):
            return self._forward_fused(V, out=out, batch_index=batch_index, gather=gather)
        if out is not None or batch_index is not None or gather is not None:
            raise NotImplementedError("out= / batch_index= / gather= are supported on the linked bf16 path only")
        V = [v.materialize() if isinstance(v, DeferredProjection) else v for v in V]
        if _needs_grad(self, *V):
            att = self.attention
            pe = self.pe if self.positional_embedding and self.averagetoken else None
            return _MixFn.apply(self, _compute_dtype(V[0]), None, None, self.Q, att.q_proj_weight, att.k_proj_weight, att.in_proj_bias, pe, *V)
        return self._forward_tokens(V)

    def _forward_assembled(self, V, asm: "_Assembly", batch_index: Optional[torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
        """(embedding buffer with the prefix in its slot, weights) through the autograd Functions (MervFusion.forward_multimodal): the fused
        training step when it covers the configuration, module by module otherwise (bf16 or fp32, any averagetoken / pe / token layout)."""
        deferred = all(isinstance(v, DeferredProjection) for v in V)
        train = _needs_grad(self, asm.emb, *[t for v in V for t in ((v.features,) if isinstance(v, DeferredProjection) else (v,))],
                            *[t for v in V if isinstance(v, DeferredProjection) for t in v.projector.parameters()])
        if deferred and train and self._can_fuse_training(V):
            return self._forward_fused_train(V, batch_index=batch_index, asm=asm)
        V = _materialize(V, batch_index)
        att = self.attention
        pe = self.pe if self.positional_embedding and self.averagetoken else None
        return _MixFn.apply(self, _compute_dtype(V[0]), asm, asm.emb, self.Q, att.q_proj_weight, att.k_proj_weight, att.in_proj_bias, pe, *V)

    def _forward_tokens(self, V: Sequence[torch.Tensor], rowdots=None) -> Tuple[torch.Tensor, torch.Tensor]:
        dtype = _compute_dtype(V[0])
        V = [v if v.dtype == dtype else v.to(dtype) for v in V]
        u = self.query_vector(dtype)  # [K] (averagetoken=True) or [T*K] (averagetoken=False: the key is the flattened token block)
        if rowdots is not None:
            scores = ops.scores_from_partials(rowdots, None, V[0].shape[0], self.token_length)
        else:
            scores = ops.scores_from_tokens(V, u, self.token_length, per_token_u=not self.averagetoken,
                                            consts=self._pe_consts(dtype), mean=self.averagetoken)
        out, weights = ops.softmax_mix(V, self.token_length, scores=scores)
        return out, weights.to(dtype)

    def _can_fuse(self, V: Sequence[DeferredProjection]) -> bool:
        if len(V) > 4 or any(v.dtype != torch.bfloat16 for v in V) or not self.averagetoken:
            return False
        if any(v.shape[1] != self.token_length for v in V):
            return False
        # one pool launch / one GEMM row space for all encoders: the same S x S grid everywhere (equal T*S*S alone would also admit
        # e.g. 16 x 8 x 8 next to 4 x 16 x 16, which the module-by-module path handles)
        if len({v.projector.output_size for v in V}) != 1:
            return False
        return all(len(v.projector.layers()) >= 1 for v in V)

    def _can_fuse_training(self, V: Sequence[DeferredProjection]) -> bool:
        """The fused backward (_FusedLinearFn) covers what MERV constructs (merv.py:152-163,214-216): single-Linear projectors with
        bias in front of the averagetoken mixer without positional embedding, bf16 compute, frozen features."""
        if not self._can_fuse(V) or self.positional_embedding or type(self) is not CrossAttentionAdapterLearnableQuery:
            return False
        for v in V:
            layers = v.projector.layers()
            if len(layers) != 1 or layers[0][0].bias is None or v.features.requires_grad:
                return False
        return self.attention.in_proj_bias is not None

    def _forward_fused_train(self, V: Sequence[DeferredProjection], batch_index=None, asm=None) -> Tuple[torch.Tensor, torch.Tensor]:
        dtype = torch.bfloat16
        projs = [v.projector for v in V]
        xs = [v.features.detach() for v in V]
        xs = [x if x.dtype == dtype else x.to(dtype) for x in xs]
        xs = [x if _tma_readable(x) else x.contiguous() for x in xs]
        att = self.attention
        params = [t for p in projs for t in (p.layers()[0][0].weight, p.layers()[0][0].bias)]
        return _FusedLinearFn.apply(self, projs, xs, batch_index, asm, None if asm is None else asm.emb, self.Q, att.q_proj_weight,
                                    att.k_proj_weight, att.in_proj_bias, *params)

    # ---- fused pipeline ------------------------------------------------------------------------------------
    def _fused_stage1(self, projs, xs, vcs, dtype, max_ctas: int = 0, batch_index=None):
        """pool (+ hidden layers) -> (A operands of the last layer, score partials)."""
        frames, size = [p.output_frames for p in projs], projs[0].output_size
        if all(len(p.layers()) == 1 for p in projs):
            # scores straight from the pool kernel: u . y = v . pooled + c for the affine projector
            return ops.pool3d(xs, frames, size, score_vecs=[vc[0] for vc in vcs], max_ctas=max_ctas, batch_index=batch_index)
        pooled, _ = ops.pool3d(xs, frames, size, max_ctas=max_ctas, batch_index=batch_index)
        acts, partials = [], []
        for p, x, (v, _) in zip(projs, pooled, vcs):
            h, rd = _run_layers(x, p.layers()[:-1], p._cast_cache, dtype, last_rowdot_vec=v)
            acts.append(h)
            partials.append(rd)
        return acts, partials

    def _forward_fused(self, V: Sequence[DeferredProjection], out: Optional[torch.Tensor] = None,
                       batch_index: Optional[torch.Tensor] = None, gather=None) -> Tuple[torch.Tensor, torch.Tensor]:
        """pool (one launch) -> hidden layers -> scores -> one tcgen05 GEMM with the mix in its epilogue.

        `out`: optional [B, T, K] bf16 view (any batch stride) the prefix is written into, e.g. the prefix slot of the
        multimodal embedding buffer (merv.py:633-640).  `batch_index`: optional int32 [B'] gather of the input videos
        (`multimodal_indices`, merv.py:572) fused into the pool kernel's loads.
        """
        dtype = torch.bfloat16
        projs = [v.projector for v in V]
        xs = [v.features if v.features.dtype == dtype else v.features.to(dtype) for v in V]
        xs = [x if _tma_readable(x) else x.contiguous() for x in xs]
        batch_index = _as_batch_index(batch_index, xs[0])
        B, T, K = (xs[0].shape[0] if batch_index is None else batch_index.numel()), self.token_length, self.llm_dim
        if out is not None:
            assert out.shape == (B, T, K) and out.dtype == dtype and out.stride(2) == 1 and out.device == xs[0].device, \
                f"out must be a bf16 [B, T, K] = {(B, T, K)} view with contiguous rows on {xs[0].device}, got {out.dtype} {tuple(out.shape)}"
        lasts = [p.layers()[-1][0] for p in projs]
        vcs = [self._affine_vec(lin, p._cast_cache, dtype) for lin, p in zip(lasts, projs)]
        if self.positional_embedding:  # score_e += u . pe[e]: folded into the per-encoder score constants
            cpe = self._pe_consts(dtype, [vc[1] for vc in vcs])
            vcs = [(vc[0], cpe[e:e + 1]) for e, vc in enumerate(vcs)]
        biases = [p._cast_cache.get(lin.bias, dtype) for lin, p in zip(lasts, projs)]
        Ws = [p._cast_cache.get(lin.weight, dtype) for lin, p in zip(lasts, projs)]
        if gather is not None:
            # fused all-gather (merv_b200.parallel.SymmetricPrefixBuffer): every output tile is also stored into this rank's
            # block of the other ranks' buffers over NVLink while the GEMM is still running; returns the WHOLE batch's prefixes
            assert out is None and B == gather.batch_per_rank and T * K * 2 * B == gather.block_bytes
            acts, partials = self._fused_stage1(projs, xs, vcs, dtype, batch_index=batch_index)
            scores = ops.scores_from_partials(partials, [vc[1] for vc in vcs], B, T)
            weights, bias_mix = ops.softmax_weights(scores, biases, K)
            gather.barrier()  # every rank has finished reading the previous contents of the buffers
            mc = gather.multicast_block_ptr() if hasattr(gather, "multicast_block_ptr") else 0
            if mc:  # one multimem.st per output byte, replicated by the NVSwitch into every rank's buffer (the local one included)
                ops.fused_linear_mix(acts, Ws, weights, bias_mix, T, out=gather.local_block(), multicast_out_ptr=mc)
            else:
                ops.fused_linear_mix(acts, Ws, weights, bias_mix, T, out=gather.local_block(), peer_out_ptrs=gather.peer_block_ptrs())
            gather.barrier()  # every rank's stores have landed
            return gather.buf, weights.to(dtype)
        timer = ops._timer
        if all(len(p.layers()) == 1 for p in projs) and (timer is None or not timer.timing) and (out is None or out.dim() == 3):
            plan = self._fused_plan(projs, xs, vcs, Ws, biases, B)
            self.__dict__["_last_plan"] = plan
            return plan.run(xs, out, batch_index)
        acts, partials = self._fused_stage1(projs, xs, vcs, dtype, batch_index=batch_index)
        scores = ops.scores_from_partials(partials, [vc[1] for vc in vcs], B, T)
        weights, bias_mix = ops.softmax_weights(scores, biases, K)
        if out is not None:
            assert out.shape == (B, T, K), f"out must be [B, T, K] = {(B, T, K)}, got {tuple(out.shape)}"
            ops.fused_linear_mix(acts, Ws, weights, bias_mix, T, out=out)
            return out, weights.to(dtype)
        res = ops.fused_linear_mix(acts, Ws, weights, bias_mix, T)
        return res.view(B, T, K), weights.to(dtype)


    def _fused_plan(self, projs, xs, vcs, Ws, biases, B) -> "ops.FusedLinearPlan":
        """One cached single-call plan per (shapes, strides, stream).  A plan owns ~B x 7.3 MB of workspaces, so a new parameter
        version (an optimizer step between two eval passes) re-binds the existing plan's pointers instead of building another."""
        key = (B, tuple((tuple(x.shape), x.stride()) for x in xs), *_stream_key(xs[0].device))
        ptag = (tuple((id(vc[0]), vc[1].data_ptr()) for vc in vcs), tuple(w.data_ptr() for w in Ws),
                tuple(None if b is None else b.data_ptr() for b in biases))
        plans = self.__dict__.setdefault("_plans", {})
        hit = plans.get(key)
        if hit is None:
            if len(plans) >= 4:  # shapes rarely change; keep the cache (and its workspaces) small
                plans.clear()
            plan = ops.FusedLinearPlan(xs, [p.output_frames for p in projs], projs[0].output_size, [vc[0] for vc in vcs],
                                       [vc[1] for vc in vcs], Ws, biases, B, xs[0].shape[0])
            plans[key] = (ptag, plan)
            return plan
        if hit[0] != ptag:
            hit[1].rebind([vc[0] for vc in vcs], [vc[1] for vc in vcs], Ws, biases)
            plans[key] = (ptag, hit[1])
        return hit[1]

    def invalidate_caches(self) -> None:
        """Drop every cached derived quantity (u, v_e, cast weights, plans).  Staleness is detected through ``Tensor._version``,
        which an update through ``.data`` (``p.data.mul_()``) or a raw-pointer write does not bump: call this after such an update."""
        self._u_cache.clear()
        self._vc_cache.clear()
        self._cast_cache = _CastCache()
        self.__dict__.pop("_plans", None)
        self.__dict__.pop("_last_plan", None)


class ScalarAdapter(_LinkedMixer):
    """One learnable scalar per encoder, softmax-normalised, the same mix for every video (nn_utils.py:524-537;
    feature_fusion == "scalar", merv.py:224-225).  Like the reference it always holds 4 scalars.

    Training: linked 3d-avg / avg pools with single-Linear projectors (bf16, T % 64 == 0) take the fused forward with a backward that keeps
    only the pooled tokens (_FusedScalarLinearFn); everything else trains module by module through _ScalarMixFn.  Whether linked
    projectors hand their input over at all is _LinkedMixer's policy (``fused_training``)."""

    def __init__(self, num_encoder=4) -> None:
        super().__init__()
        self.scalar = torch.nn.Parameter(torch.randn(4))
        self.fused_training: Optional[bool] = None  # see _LinkedMixer

    def forward(self, projected_patch_embeddings):
        V = projected_patch_embeddings
        E = len(V)
        assert E == self.scalar.numel(), f"ScalarAdapter holds {self.scalar.numel()} scalars, got {E} encoders (nn_utils.py:527,535)"
        proj_params = [t for v in V if isinstance(v, DeferredProjection) for t in v.projector.parameters()]
        if _needs_grad(self, *[v for v in V if isinstance(v, torch.Tensor)], *proj_params):
            return self._forward_train(V)
        linked = all(isinstance(v, DeferredProjection) for v in V)
        first = V[0].features if linked else V[0]
        B = first.shape[0]
        scores = self.scalar.detach().float().reshape(1, E).expand(B, E).contiguous()  # softmax happens in the kernels
        if linked and all(v.dtype == torch.bfloat16 and len(v.projector.layers()) == 1 for v in V) and \
                len({(v.projector.output_size, v.shape[1]) for v in V}) == 1:
            # affine projectors: out = sum_e w_e (P_e W_e^T + b_e) in one tcgen05 GEMM, Y_e never written
            dtype = torch.bfloat16
            projs = [v.projector for v in V]
            xs = [v.features if v.features.dtype == dtype else v.features.to(dtype) for v in V]
            pooled, _ = ops.pool3d(xs, [p.output_frames for p in projs], projs[0].output_size)
            lasts = [p.layers()[-1][0] for p in projs]
            weights, bias_mix = ops.softmax_weights(scores, [p._cast_cache.get(l.bias, dtype) for l, p in zip(lasts, projs)], lasts[0].out_features)
            T = V[0].shape[1]
            out = ops.fused_linear_mix(pooled, [p._cast_cache.get(l.weight, dtype) for l, p in zip(lasts, projs)], weights, bias_mix, T)
            return out.view(B, T, -1), weights[:1].to(dtype)
        V = [v.materialize() if isinstance(v, DeferredProjection) else v for v in V]
        dtype = _compute_dtype(V[0])
        V = [v if v.dtype == dtype else v.to(dtype) for v in V]
        out, weights = ops.softmax_mix(V, V[0].shape[1], scores=scores)
        return out, weights[:1].to(dtype)

    def _forward_assembled(self, V, asm: "_Assembly", batch_index: Optional[torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
        """(embedding buffer with the prefix in its slot, weights), as CrossAttentionAdapterLearnableQuery._forward_assembled."""
        E = len(V)
        assert E == self.scalar.numel(), f"ScalarAdapter holds {self.scalar.numel()} scalars, got {E} encoders (nn_utils.py:527,535)"
        proj_params = [t for v in V if isinstance(v, DeferredProjection) for t in v.projector.parameters()]
        if _needs_grad(self, asm.emb, *[v for v in V if isinstance(v, torch.Tensor)], *proj_params) and asm.idx.numel() and self._can_fuse_training(V):
            return self._forward_train(V, batch_index=batch_index, asm=asm)
        V = _materialize(V, batch_index)
        if len({tuple(v.shape) for v in V}) != 1:
            raise ValueError("the ScalarAdapter needs every encoder at one [B, T, K] shape to mix into the embedding buffer (the reference "
                             f"stacks them, nn_utils.py:535), got {[tuple(v.shape) for v in V]}")
        return _ScalarMixFn.apply(self.scalar, _compute_dtype(V[0]), asm, asm.emb, *V)

    def _can_fuse_training(self, V) -> bool:
        """The fused backward (_FusedScalarLinearFn) covers single-Linear projectors with bias on one pooled grid, bf16 compute, token
        counts that are a multiple of 64 (a k-block of merv_wgrad_video never spans two videos), frozen features, at least one video."""
        if not all(isinstance(v, DeferredProjection) for v in V) or any(v.dtype != torch.bfloat16 for v in V):
            return False
        if len({(v.projector.output_size, v.shape[1]) for v in V}) != 1 or V[0].shape[1] % 64 or V[0].shape[0] == 0:
            return False
        for v in V:
            layers = v.projector.layers()
            if len(layers) != 1 or layers[0][0].bias is None or v.features.requires_grad:
                return False
        return True

    def _forward_train(self, V, batch_index=None, asm=None) -> Tuple[torch.Tensor, torch.Tensor]:
        if self._can_fuse_training(V):
            dtype = torch.bfloat16
            projs = [v.projector for v in V]
            xs = [v.features.detach() for v in V]
            xs = [x if x.dtype == dtype else x.to(dtype) for x in xs]
            xs = [x if _tma_readable(x) else x.contiguous() for x in xs]
            params = [t for p in projs for t in (p.layers()[0][0].weight, p.layers()[0][0].bias)]
            return _FusedScalarLinearFn.apply(self, projs, xs, batch_index, asm, None if asm is None else asm.emb, self.scalar, *params)
        V = [v.materialize() if isinstance(v, DeferredProjection) else v for v in V]
        if len({tuple(v.shape) for v in V}) != 1:
            raise ValueError("training the ScalarAdapter needs every encoder at one [B, T, K] shape (the reference stacks them, "
                             f"nn_utils.py:535), got {[tuple(v.shape) for v in V]}")
        return _ScalarMixFn.apply(self.scalar, _compute_dtype(V[0]), None, None, *V)


class ConcatChannelFusion(LinearProjector):
    """feature_fusion == "concat_channel" (merv.py:217-218): ``LinearProjector(E * llm_dim, llm_dim)`` applied to the
    channel-wise concatenation of the projected tokens (merv.py:603-606).  Same parameters / state-dict keys as the
    reference's LinearProjector (``feature_fusion.projector.{weight,bias}``).

    ``forward(tensor)`` is the reference call (the glue concatenated already).  ``forward(list)`` takes the per-encoder
    tokens and runs sum_e Y_e W[:, e-th block]^T + b as ONE K-segmented tcgen05 GEMM: the [B, T, E * llm_dim] tensor is
    never built (saves writing and re-reading 2 x E x 8.4 MB per video at merv-full sizes)."""

    def __init__(self, num_encoder: int, llm_dim: int) -> None:
        super().__init__(num_encoder * llm_dim, llm_dim)
        self.num_encoder = num_encoder

    def forward(self, projected_patch_embeddings):
        V = projected_patch_embeddings
        if isinstance(V, torch.Tensor):
            return super().forward(V)
        V = [v.materialize() if isinstance(v, DeferredProjection) else v for v in V]
        lin = self.projector
        assert sum(v.shape[-1] for v in V) == lin.in_features, f"concat_channel expects {lin.in_features} channels in total"
        dtype = _compute_dtype(V[0])
        segmented = (dtype == torch.bfloat16 and len(V) <= MAX_SEGMENTS and all(v.shape[-1] % 8 == 0 for v in V)
                     and not _needs_grad(self, *V))
        if not segmented or V[0].numel() == 0:  # fp32 parity path / training / > 4 encoders: concatenate as the reference does
            return super().forward(torch.concat(V, -1))
        if not hasattr(self, "_cast_cache"):
            self._cast_cache = _CastCache()
        V = [v if v.dtype == dtype else v.to(dtype) for v in V]
        return ops.concat_linear(V, self._cast_cache.get(lin.weight, dtype), self._cast_cache.get(lin.bias, dtype))


class ConcatChannelLNFusion(nn.Sequential):
    """feature_fusion == "concat_channel_ln" (merv.py:219-223): ``Sequential(LayerNorm(E * llm_dim), LinearProjector(E * llm_dim,
    llm_dim))`` applied to the channel-wise concatenation of the projected tokens (merv.py:603-606).  Same module tree as the
    reference, hence the same state-dict keys (``feature_fusion.0.{weight,bias}``, ``feature_fusion.1.projector.{weight,bias}``).

    ``forward(tensor)`` is the reference call.  ``forward(list)`` takes the per-encoder tokens: the LayerNorm kernel reads them as
    row segments and writes the NORMALISED concatenation once (the un-normalised one is never built), then one plain tcgen05 GEMM."""

    def __init__(self, num_encoder: int, llm_dim: int) -> None:
        super().__init__(nn.LayerNorm(num_encoder * llm_dim), LinearProjector(num_encoder * llm_dim, llm_dim))
        self.num_encoder = num_encoder

    def forward(self, projected_patch_embeddings):
        V = projected_patch_embeddings
        ln, proj = self[0], self[1]
        segs = [V] if isinstance(V, torch.Tensor) else [v.materialize() if isinstance(v, DeferredProjection) else v for v in V]
        _require_device(segs[0])
        lin = proj.projector
        assert sum(v.shape[-1] for v in segs) == lin.in_features, f"concat_channel_ln expects {lin.in_features} channels in total"
        dtype = _compute_dtype(segs[0])
        if not hasattr(self, "_cast_cache"):
            self._cast_cache = _CastCache()
        cache = self._cast_cache
        segs = [v if v.dtype == dtype else v.to(dtype) for v in segs]
        if segs[0].numel() == 0:
            return torch.empty((*segs[0].shape[:-1], lin.out_features), dtype=dtype, device=segs[0].device)
        if _needs_grad(self, *segs):  # training: concatenate as the reference does, one autograd node with the hand-written backward
            x = segs[0] if len(segs) == 1 else torch.concat(segs, -1)
            y, _ = _run_layers(x, [(lin, ACT_NONE)], cache, dtype, train=True, ln=ln)
            return y
        vec = 8 if dtype == torch.bfloat16 else 4
        if len(segs) > 8 or any(v.shape[-1] % vec for v in segs):
            segs = [torch.concat(segs, -1)]
        x = ops.layernorm(segs, cache.get(ln.weight, dtype), cache.get(ln.bias, dtype), ln.eps)
        y, _ = ops.linear_bias_act(x, cache.get(lin.weight, dtype), cache.get(lin.bias, dtype), ACT_NONE)
        return y


# ------------------------------------------------------------------------------------------------------------
# linking: the fused pipeline behind the unchanged MERV.forward glue
# ------------------------------------------------------------------------------------------------------------
def link_fused(projectors: Sequence[AveragePooling3DProjector], feature_fusion: CrossAttentionAdapterLearnableQuery) -> None:
    """Make ``projector(x)`` return a DeferredProjection that ``feature_fusion`` turns into the fused pipeline."""
    for p in projectors:
        p._linked_fusion = weakref.ref(feature_fusion)


def unlink(projectors: Sequence[AveragePooling3DProjector]) -> None:
    for p in projectors:
        p._linked_fusion = None


class MervFusion(nn.Module):
    """projectors + feature_fusion as one module: ``forward(patch_features) -> (prefix [B,T,K], weights [B,E])``.

    Restates the glue of merv/models/vidlms/merv.py:587-589,607-609 with the sub-module names MERV uses
    (``projectors``, ``feature_fusion``) so ``state_dict()`` keys match a MERV checkpoint's.
    """

    def __init__(self, projectors: Sequence[AveragePooling3DProjector], feature_fusion: Optional[nn.Module],
                 fused: bool = True, fusion_type: Optional[str] = None, fused_training: Optional[bool] = None) -> None:
        super().__init__()
        self.projectors = nn.ModuleList(projectors)
        self.feature_fusion = feature_fusion
        if fused_training is not None:  # force the training step onto / off the fused forward + backward (None: automatic)
            assert not fused_training or (fused and isinstance(feature_fusion, _LinkedMixer)), \
                "fused_training needs a linked learnable-query or scalar mixer"
            if isinstance(feature_fusion, _LinkedMixer):
                feature_fusion.fused_training = fused_training
        # the parameter-free fusions of merv.py:598-601: "first" (encoder 0 only) and "concat" (token-wise concatenation)
        self.fusion_type = fusion_type
        if feature_fusion is None:
            assert fusion_type in ("first", "concat"), "feature_fusion=None needs fusion_type 'first' or 'concat' (merv.py:598-601)"
        # concat_channel(_ln) consume the projected tokens themselves
        elif fused and not isinstance(feature_fusion, (ConcatChannelFusion, ConcatChannelLNFusion)):
            link_fused(self.projectors, self.feature_fusion)

    def _forward_token_concat(self, patch_features: Sequence[torch.Tensor]) -> torch.Tensor:
        """feature_fusion == "concat" (merv.py:600-601): ``torch.concat(projected, 1)`` -> [B, sum_e T_e, K].  For bf16 affine
        projectors with tile-aligned token counts every projector's GEMM stores straight into its slice of the result through
        the batch-strided TMA-store map (no concat copy); otherwise the projected tokens are copied into place."""
        projs = list(self.projectors)
        Ts = [p.output_frames * p.output_size**2 for p in projs]
        x0 = patch_features[0]
        dtype = _compute_dtype(x0)
        B, K = x0.shape[0], projs[0].llm_dim
        out = torch.empty((B, sum(Ts), K), dtype=dtype, device=x0.device)
        t0 = 0
        for p, x, T in zip(projs, patch_features, Ts):
            dst = out[:, t0:t0 + T]
            t0 += T
            if B == 0:
                continue
            direct = (dtype == torch.bfloat16 and len(p.layers()) == 1 and T % 128 == 0 and not _needs_grad(p, x)
                      and p.layers()[0][0].bias is not None)
            if not direct:
                dst.copy_(p._forward_unfused(x))
                continue
            xb = x.detach() if x.dtype == dtype else x.detach().to(dtype)
            (pooled,), _ = ops.pool3d([xb], [p.output_frames], p.output_size)
            lin = p.layers()[0][0]
            # one encoder with scale softmax([0]) == 1 and bias rows 1 * bias: the batch-strided form of the fused GEMM
            ones, bias_rows = ops.softmax_weights(torch.zeros((B, 1), dtype=torch.float32, device=x.device),
                                                  [p._cast_cache.get(lin.bias, dtype)], K)
            ops.fused_linear_mix([pooled], [p._cast_cache.get(lin.weight, dtype)], ones, bias_rows, T, out=dst)
        return out

    @classmethod
    def build(cls, vision_dims: Sequence[int], llm_dim: int, output_frames: Sequence[int], projector_token_length: int = 64,
              mlp_type: str = "linear", text_embedding_dim: int = 3072, seed: Optional[int] = None, fused: bool = True) -> "MervFusion":
        """Construct as MERV.__init__ does (merv.py:87,110-163,214-216), including the projector-consistency seed."""
        if seed is not None:
            torch.manual_seed(seed)
        size = int(projector_token_length**0.5)
        assert projector_token_length == size**2, "projector_token_length should be square number"
        projs = [AveragePooling3DProjector(c, llm_dim, output_frames=t, output_size=size, mlp_type=mlp_type)
                 for c, t in zip(vision_dims, output_frames)]
        lengths = {p.output_token_length * p.output_frame_length for p in projs}
        assert len(lengths) == 1, f"Output token length is not consistent across all projectors! {sorted(lengths)}"
        fusion = CrossAttentionAdapterLearnableQuery(embed_dim=text_embedding_dim, llm_dim=llm_dim, token_length=lengths.pop(),
                                                     averagetoken=True, num_encoder=len(projs))
        return cls(projs, fusion, fused=fused)

    @classmethod
    def from_config(cls, vision_dims: Sequence[int], llm_dim: int, temporal_resolutions: Sequence[int], arch_specifier: str = "gelu-mlp",
                    feature_fusion: Optional[str] = None, projector_token_length: int = 64, visual_feature_length: int = 512,
                    pre_proj_layernorm: bool = False, text_embedding_dim: int = 3072, num_patches: Optional[Sequence[int]] = None,
                    seed: Optional[int] = -1, fused: bool = True, fused_training: Optional[bool] = None) -> "MervFusion":
        """Build the projectors and the feature-fusion module from the reference's OWN config strings, as ``MERV.__init__`` does
        (merv.py:87-227; config surface ``conf/models.py:28-43``): same parsing of ``arch_specifier`` (suffix = projector type,
        ``+``-separated resampler, optional ``frameN`` temporal factor) and ``feature_fusion``, same construction order — hence the
        same RNG consumption under the projector-consistency seed ``torch.manual_seed(video_backbones[0].embed_dim)`` (merv.py:87;
        ``seed=-1`` reproduces it, ``None`` leaves the RNG alone) — same consistency asserts and the same exceptions.

        ``vision_dims[i]`` / ``temporal_resolutions[i]`` / ``num_patches[i]`` stand for ``video_backbones[i].embed_dim`` /
        ``.temporal_resolution`` / ``.num_patches``.  The ``conv`` resampler (timm RegStage blocks) is outside the accelerated path
        (DESIGN.md "Out of scope") and raises NotImplementedError instead of falling back; the ``query_mlp`` mixer is constructed as the
        reference constructs it (merv.py:211-212) and, as in the reference (no forward branch, merv.py:598-612), raises when called."""
        import re
        from functools import partial

        if seed is not None:
            torch.manual_seed(vision_dims[0] if seed == -1 else seed)  # merv.py:87
        # merv.py:89-105
        if arch_specifier.endswith("linear"):
            mlp_type, Projector = "linear", LinearProjector
        elif arch_specifier.endswith("fused-gelu-mlp"):
            mlp_type, Projector = "fused-gelu-mlp", FusedMLPProjector
        elif arch_specifier.endswith("gelu-mlp"):
            mlp_type, Projector = "gelu-mlp", MLPProjector
        elif arch_specifier.endswith("none"):
            mlp_type, Projector = "none", None  # "will get overriden later" (merv.py:100-103): only valid with a resampler
        else:
            raise ValueError(f"MERV with `{arch_specifier = }` is not supported!")
        # merv.py:107-150
        tokens_resampled, factor = False, 1
        size = int(projector_token_length**0.5)
        assert projector_token_length == size**2, "projector_token_length should be square number"
        parts = arch_specifier.split("+")

        def frame_factor() -> int:
            return int(re.search(r"frame(\d+)", arch_specifier).group(1)) if "frame" in arch_specifier else 1

        if "avg" in parts:
            tokens_resampled, Projector = True, partial(AveragePoolingProjector, output_size=size)
        elif "attntv" in parts:
            tokens_resampled, Projector = True, partial(AttentivePooler, num_query_tokens=projector_token_length, num_heads=8)
        elif "conv" in parts:
            raise NotImplementedError("the `conv` resampler (ConvolutionalProjector, nn_utils.py:249-303) is not part of the accelerated path")
        elif "3davg" in parts:
            factor = frame_factor()
            tokens_resampled, Projector = True, partial(AveragePooling3DProjector, output_size=size)
        elif "3dconv" in parts:  # merv.py:142-150
            factor = frame_factor()
            tokens_resampled, Projector = True, partial(Convolutional3DProjector, output_size=size)
        # merv.py:152-172
        if tokens_resampled:
            projs = [Projector(c, llm_dim, output_frames=t // factor, mlp_type=mlp_type) for c, t in zip(vision_dims, temporal_resolutions)]
        else:
            if Projector is None:
                raise ValueError(f"MERV with `{arch_specifier = }` is not supported!")  # an nn.Identity() instance is not constructible
            projs = [Projector(c, llm_dim, pre_proj_layernorm=pre_proj_layernorm) for c in vision_dims]
        # merv.py:174-208
        if len(vision_dims) > 1:
            if tokens_resampled:
                assert all(p.output_token_length * p.output_frame_length in [1, visual_feature_length] for p in projs), (
                    "Output token length is not consistent across all projectors!"
                    f" visual_feature_length={visual_feature_length}."
                    f" {[(p.__class__.__name__, p.output_token_length, 'X', p.output_frame_length) for p in projs]}")
            else:
                assert all(getattr(p, "output_token_length", 1) * t in [1, visual_feature_length] for p, t in zip(projs, temporal_resolutions)), (
                    "Output token length is not consistent across all projectors!" f" visual_feature_length={visual_feature_length}.")
        else:
            if tokens_resampled:
                correct_length = projs[0].output_token_length * projs[0].output_frame_length
            else:
                assert num_patches is not None, "a single un-resampled encoder needs num_patches (video_backbones[0].num_patches, merv.py:200)"
                correct_length = num_patches[0]
            visual_feature_length = correct_length
        # merv.py:211-227
        E = len(vision_dims)
        if feature_fusion == "query_mlp":
            # merv.py:211-212 constructs it (so checkpoints carry its parameters) but MERV.forward has no branch for it (merv.py:598-612):
            # same module tree / init here, and forward raises what the reference raises
            ff = MLPProjector(3072, E)
        elif feature_fusion == "cross_attention_avg_lq":
            ff = CrossAttentionAdapterLearnableQuery(embed_dim=3072, llm_dim=llm_dim, token_length=visual_feature_length, averagetoken=True)
        elif feature_fusion == "concat_channel":
            ff = ConcatChannelFusion(E, llm_dim)
        elif feature_fusion == "concat_channel_ln":
            ff = ConcatChannelLNFusion(E, llm_dim)
        elif feature_fusion == "scalar":
            ff = ScalarAdapter(E)
        else:
            ff = None
            if feature_fusion not in ("first", "concat"):  # merv.py:610-612
                print(f'feature_fusion "{feature_fusion}" doesn\'t exist')
                raise NotImplementedError
        linkable = fused and tokens_resampled and all(isinstance(p, AveragePooling3DProjector) for p in projs) and \
            isinstance(ff, (CrossAttentionAdapterLearnableQuery, ScalarAdapter))
        m = cls(projs, ff, fused=linkable, fusion_type=feature_fusion if ff is None else None,
                fused_training=fused_training if linkable else None)
        m.arch_specifier, m.feature_fusion_type, m.tokens_resampled = arch_specifier, feature_fusion, tokens_resampled
        m.visual_feature_length, m.text_embedding_dim = visual_feature_length, text_embedding_dim
        return m

    # ---- small-batch fast path: skip the per-module Python glue when nothing changed since the last call -------------
    def _param_tag(self):
        ff = self.feature_fusion
        ps = [ff.Q, ff.attention.q_proj_weight, ff.attention.k_proj_weight, ff.attention.in_proj_bias]
        if ff.positional_embedding:
            ps.append(ff.pe)
        for p in self.projectors:
            for lin, _ in p.layers():
                ps += [lin.weight] + ([lin.bias] if lin.bias is not None else [])
        if any(_is_volatile(t) for t in ps):  # FSDP views: contents change behind a constant (data_ptr, version)
            return None
        return tuple((t.data_ptr(), _version(t)) for t in ps)

    def _fast_forward(self, xs, out, batch_index):
        """Re-run the cached single-call plan (ops.FusedLinearPlan) if shapes, strides, stream and every parameter version
        are unchanged; returns None when the general path has to (re)build it.  Saves ~50 us of Python per call, which is
        most of the cost at B = 1."""
        ff = self.feature_fusion
        timer = ops._timer
        if (timer is not None and timer.timing) or not isinstance(ff, CrossAttentionAdapterLearnableQuery):
            return None
        x0 = xs[0]
        if not x0.is_cuda or x0.shape[0] == 0 or any(x.dtype != torch.bfloat16 for x in xs) or (out is not None and out.dim() != 3):
            return None
        # the plan's descriptor records the strides it was built with: only inputs the kernels read IN PLACE may re-run it
        # (anything else is copied to contiguous memory by the general path, whose plan then describes the copy)
        if not all(_tma_readable(x) for x in xs):
            return None
        batch_index = _as_batch_index(batch_index, x0)
        key = (tuple((x.shape, x.stride()) for x in xs), None if batch_index is None else batch_index.numel(), *_stream_key(x0.device))
        cache = self.__dict__.setdefault("_fast", {})
        hit = cache.get(key)
        tag = self._param_tag()
        if tag is None:
            return None
        if hit is not None and hit[0] == tag:
            return hit[1].run(xs, out, batch_index, xs_checked=True)  # `key` holds exactly what run() would re-check about xs
        # general path once; remember the plan it used (if it took the single-call route)
        ff.__dict__["_last_plan"] = None
        projected = [proj(x) for proj, x in zip(self.projectors, xs)]
        res = ff(projected, out=out, batch_index=batch_index) if (out is not None or batch_index is not None) else ff(projected)
        plan = ff.__dict__.get("_last_plan")
        if plan is not None and all(isinstance(p.projector, LinearProjector) for p in self.projectors):
            if len(cache) >= 4:
                cache.clear()
            cache[key] = (tag, plan)
        return res

    def invalidate_caches(self) -> None:
        """See CrossAttentionAdapterLearnableQuery.invalidate_caches (needed after parameter updates that bypass ``_version``)."""
        self.__dict__.pop("_fast", None)
        for p in self.projectors:
            if hasattr(p, "_cast_cache"):
                p._cast_cache = _CastCache()
        if hasattr(self.feature_fusion, "invalidate_caches"):
            self.feature_fusion.invalidate_caches()

    def forward(self, patch_features: Sequence[torch.Tensor], out: Optional[torch.Tensor] = None,
                batch_index: Optional[torch.Tensor] = None, gather=None) -> Tuple[torch.Tensor, torch.Tensor]:
        if self.feature_fusion is None:  # merv.py:598-601: "first" / "concat", no module and no mixing weights
            assert out is None and batch_index is None and gather is None, "'first' / 'concat' support the plain call only"
            if self.fusion_type == "first":
                p0 = self.projectors[0]
                return (p0._forward_unfused(patch_features[0]) if hasattr(p0, "_forward_unfused") else p0(patch_features[0])), None
            if not all(isinstance(p, AveragePooling3DProjector) for p in self.projectors):  # un-resampled / attntv projectors
                ys = [p(x) for p, x in zip(self.projectors, patch_features)]
                out_cat = torch.empty((ys[0].shape[0], sum(y.shape[1] for y in ys), ys[0].shape[2]), dtype=ys[0].dtype, device=ys[0].device)
                t0 = 0
                for y in ys:  # merv.py:600-601 (token-wise concatenation: a copy, no arithmetic)
                    out_cat[:, t0:t0 + y.shape[1]].copy_(y)
                    t0 += y.shape[1]
                return out_cat, None
            return self._forward_token_concat(patch_features), None
        if getattr(self, "feature_fusion_type", None) == "query_mlp":  # merv.py:610-612: constructed, but no forward branch in the reference
            print(f'feature_fusion "{self.feature_fusion_type}" doesn\'t exist')
            raise NotImplementedError
        if isinstance(self.feature_fusion, (ConcatChannelFusion, ConcatChannelLNFusion)):  # merv.py:603-606: no mixing weights
            assert out is None and batch_index is None and gather is None, "concat_channel supports the plain call only"
            return self.feature_fusion([proj(x) for proj, x in zip(self.projectors, patch_features)]), None
        if gather is not None:  # fused all-gather of the prefixes over NVLink (parallel.SymmetricPrefixBuffer)
            projected = [proj(x) for proj, x in zip(self.projectors, patch_features)]
            return self.feature_fusion(projected, batch_index=batch_index, gather=gather)
        if not torch.is_grad_enabled() and len(self.projectors) and getattr(self.projectors[0], "_linked_fusion", None) is not None:
            res = self._fast_forward(patch_features, out, batch_index)
            if res is not None:
                return res
        projected = [proj(x) for proj, x in zip(self.projectors, patch_features)]
        if out is None and batch_index is None:
            return self.feature_fusion(projected)
        return self.feature_fusion(projected, out=out, batch_index=batch_index)

    def _slot_inference(self, patch_features: Sequence[torch.Tensor], input_embeddings: torch.Tensor) -> bool:
        """Whether the linked bf16 inference path (the cached single-call plan, _forward_fused with ``out=``) writes the prefix: autograd
        records nothing, the learnable-query mixer fuses these inputs.  Everything else assembles the embeddings inside the mixer's autograd
        Function (_Assembly): training, fp32, and the module-by-module path."""
        ff = self.feature_fusion
        if not isinstance(ff, CrossAttentionAdapterLearnableQuery) or _needs_grad(self, input_embeddings, *patch_features):
            return False
        if ff.token_length % 128:  # the GEMM's batch-strided slot store works in 128-row tiles
            return False
        if any(getattr(p, "_linked_fusion", None) is None or not ff._may_defer(p) for p in self.projectors):
            return False
        return ff._can_fuse([DeferredProjection(p, x) for p, x in zip(self.projectors, patch_features)])

    def _project(self, patch_features: Sequence[torch.Tensor], batch_index: Optional[torch.Tensor]) -> list:
        """The projectors' outputs for the videos `batch_index` selects: a linked projector that hands its input over keeps the whole batch
        (the fused pool gathers in-kernel, _materialize otherwise); every other projector sees the gathered features."""
        ff = self.feature_fusion
        out = []
        for p, x in zip(self.projectors, patch_features):
            defers = getattr(p, "_linked_fusion", None) is not None and ff._may_defer(p)
            if batch_index is not None and not defers:
                x = x.index_select(0, batch_index.to(device=x.device, dtype=torch.long))
            out.append(p(x))
        return out

    def _assemble(self, patch_features: Sequence[torch.Tensor], input_embeddings: torch.Tensor, idx: Optional[torch.Tensor],
                  uni: torch.Tensor, bos: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(embedding buffer, weights) with the assembly inside the mixer's autograd Function; `idx` None = every row is multimodal."""
        ff = self.feature_fusion
        if not isinstance(ff, (CrossAttentionAdapterLearnableQuery, ScalarAdapter)):
            raise NotImplementedError("the embedding assembly covers the learnable-query and scalar mixers")
        dev = input_embeddings.device
        bi = None if idx is None else _as_batch_index(idx, patch_features[0])
        asm = _Assembly(input_embeddings, torch.arange(input_embeddings.shape[0], device=dev) if idx is None else idx.to(dev), uni, bos)
        return ff._forward_assembled(self._project(patch_features, bi), asm, bi)

    def forward_into_embeddings(self, patch_features: Sequence[torch.Tensor], input_embeddings: torch.Tensor,
                                bos_token_length: int = 1, multimodal_indices: Optional[torch.Tensor] = None):
        """Build `[BOS | visual prefix | text]` embeddings as MERV.forward does (merv.py:572,633-640) without the
        concat copy of the prefix: the buffer is allocated once, the text embeddings are copied around the prefix slot
        and the fused GEMM writes the prefix straight into it.  Returns (multimodal_embeddings, weights).
        In grad mode, in fp32 and on the module-by-module path the buffer belongs to the mixer's autograd Function: the prefix gradient is
        read from the buffer's gradient in place, and ``input_embeddings`` get theirs (rows outside ``multimodal_indices``: zeros)."""
        ff = self.feature_fusion
        if not self._slot_inference(patch_features, input_embeddings):
            idx = multimodal_indices
            uni = torch.zeros(0, dtype=torch.long, device=input_embeddings.device)
            return self._assemble(patch_features, input_embeddings, None if idx is None else idx.to(input_embeddings.device), uni,
                                  bos_token_length)
        idx = multimodal_indices
        emb = input_embeddings if idx is None else input_embeddings[idx]
        B, L, K = emb.shape
        T = ff.token_length
        buf = torch.empty((B, L + T, K), dtype=torch.bfloat16, device=emb.device)
        buf[:, :bos_token_length].copy_(emb[:, :bos_token_length])
        buf[:, bos_token_length + T:].copy_(emb[:, bos_token_length:])
        _, weights = self.forward(patch_features, out=buf[:, bos_token_length:bos_token_length + T],
                                  batch_index=None if idx is None else idx.to(torch.int32))
        return buf, weights

    def forward_multimodal(self, patch_features: Sequence[torch.Tensor], input_embeddings: torch.Tensor,
                           attention_mask: Optional[torch.Tensor] = None, labels: Optional[torch.Tensor] = None,
                           multimodal_indices: Optional[torch.Tensor] = None, bos_token_length: int = 1,
                           unimodal_indices: Optional[torch.Tensor] = None):
        """Everything MERV.forward does between the backbones and the LLM call (merv.py:572-720) for the accelerated
        configurations: gather by ``multimodal_indices``, fuse, and assemble ``fused_embeddings`` / ``fused_attention_mask``
        / ``fused_labels`` — multimodal examples first as ``[BOS | prefix | text]`` (mask True, labels IGNORE_INDEX over
        the prefix, merv.py:622-664), then the text-only examples padded at the END with T zero embeddings (mask False,
        labels IGNORE_INDEX, merv.py:668-720).  One buffer is allocated; the fused GEMM writes the prefix into it in place.

        ``patch_features[e]`` is the backbone output for the WHOLE batch (it is gathered inside the pool kernel).
        ``unimodal_indices`` may be passed to avoid the host sync the reference's Python loop (merv.py:668-672) implies.
        In grad mode, in fp32, with the scalar mixer and on the module-by-module path the buffer belongs to the mixer's autograd Function
        (_Assembly): the kernels read the prefix gradient from the buffer's gradient in place and ``input_embeddings`` get theirs.
        Returns (fused_embeddings, fused_attention_mask | None, fused_labels | None, weights)."""
        ff = self.feature_fusion
        emb = input_embeddings
        Bt, L, K = emb.shape
        dev = emb.device
        idx = torch.arange(Bt, device=dev) if multimodal_indices is None else multimodal_indices.to(dev)
        if unimodal_indices is None:
            keep = torch.ones(Bt, dtype=torch.bool, device=dev)
            keep[idx] = False
            unimodal_indices = keep.nonzero().flatten()
        uni = unimodal_indices.to(dev)
        Bm, Bu = idx.numel(), uni.numel()
        bos = bos_token_length
        whole = multimodal_indices is None
        if self._slot_inference(patch_features, emb):
            T = ff.token_length
            buf = torch.empty((Bm + Bu, L + T, K), dtype=torch.bfloat16, device=dev)
            buf[:Bm, :bos].copy_(emb[idx, :bos])
            buf[:Bm, bos + T:].copy_(emb[idx, bos:])
            if Bu:
                buf[Bm:, :L].copy_(emb[uni])
                buf[Bm:, L:].zero_()
            _, weights = self.forward(patch_features, out=buf[:Bm, bos:bos + T], batch_index=None if whole else idx.to(torch.int32))
        else:
            buf, weights = self._assemble(patch_features, emb, None if whole else idx, uni, bos)
            T = buf.shape[1] - L

        def splice(t, fill_mm, fill_uni):
            if t is None:
                return None
            res = torch.empty((Bm + Bu, L + T), dtype=t.dtype, device=t.device)
            res[:Bm, :bos] = t[idx, :bos]
            res[:Bm, bos:bos + T] = fill_mm
            res[:Bm, bos + T:] = t[idx, bos:]
            if Bu:
                res[Bm:, :L] = t[uni]
                res[Bm:, L:] = fill_uni
            return res

        return buf, splice(attention_mask, True, False), splice(labels, IGNORE_INDEX, IGNORE_INDEX), weights


_PLAIN_PROJECTORS = {"LinearProjector": LinearProjector, "MLPProjector": MLPProjector, "MLPDeepProjector": MLPDeepProjector,
                     "FusedMLPProjector": FusedMLPProjector}


def _adopt_plain_projector(ref_module: nn.Module) -> nn.Module:
    """B200 twin of a reference LinearProjector / MLPProjector / MLPDeepProjector / FusedMLPProjector sharing its submodules
    (``projector`` and the ``layernorm`` of pre_proj_layernorm), so parameters and state-dict keys are untouched."""
    cls = _PLAIN_PROJECTORS[type(ref_module).__name__]
    if isinstance(ref_module, cls):
        return ref_module
    new = cls.__new__(cls)
    nn.Module.__init__(new)
    new.projector, new.layernorm = ref_module.projector, ref_module.layernorm
    if hasattr(ref_module, "initial_projection_dim"):
        new.initial_projection_dim = ref_module.initial_projection_dim
    return new


def fsdp_wrap_policy(fused_training: Optional[bool] = None):
    """The VidLM part of the reference's FSDP auto-wrap policy (merv.py:473-485) over the B200 classes: every projector class is its
    own FSDP unit, ``feature_fusion`` folds into the root unit.  ``fused_training=True`` returns a policy that wraps NONE of them:
    projectors and adapter then share the root unit, whose parameters stay unsharded for the whole forward / backward, which is
    what the fused training step (``_FusedLinearFn``: it reads every projector's weights inside the adapter's forward) needs.
    Combine with the backbones' policies through ``_or_policy`` exactly as merv.py:487-497 does; ``patch_merv`` does that for a
    live ``MERV`` by extending its ``get_fsdp_wrapping_policy``."""
    from functools import partial

    from torch.distributed.fsdp.wrap import _module_wrap_policy

    classes = set() if fused_training else {LinearProjector, MLPProjector, FusedMLPProjector, AveragePoolingProjector, MLPDeepProjector,
                                            AveragePooling3DProjector, Convolutional3DProjector}
    return partial(_module_wrap_policy, module_classes=classes)


def _extend_fsdp_policy(vidlm: nn.Module, fused_training: Optional[bool]) -> None:
    """Make ``vidlm.get_fsdp_wrapping_policy()`` (merv.py:465-497, called by fsdp.py:208) cover the swapped-in classes."""
    orig = getattr(vidlm, "get_fsdp_wrapping_policy", None)
    if orig is None or getattr(orig, "_merv_b200_extended", False):
        return
    from functools import partial

    from torch.distributed.fsdp.wrap import _or_policy

    def get_fsdp_wrapping_policy():
        # the reference's own union stays (backbones, LLM; its projector-class entry matches nothing any more: no reference
        # projector instance is left in the module tree) and the B200 classes are added to it
        return partial(_or_policy, policies=[orig(), fsdp_wrap_policy(fused_training)])

    get_fsdp_wrapping_policy._merv_b200_extended = True
    vidlm.get_fsdp_wrapping_policy = get_fsdp_wrapping_policy


def patch_merv(vidlm: nn.Module, fused: bool = True, fused_training: Optional[bool] = None) -> nn.Module:
    """Swap a live reference ``MERV``'s hot-path modules for the B200 ones in place (parameters are shared, not copied).

    ``vidlm.projectors[i]`` (reference AveragePooling3DProjector) and ``vidlm.feature_fusion`` (reference
    CrossAttentionAdapterLearnableQuery) keep their names, so checkpoints and ``all_module_keys`` (merv.py:235) keep working, and
    ``vidlm.get_fsdp_wrapping_policy()`` (merv.py:465-497, consumed at fsdp.py:208) is extended to the B200 classes: call
    ``patch_merv`` BEFORE the FSDP wrap.  Under that policy every projector is its own FSDP unit, the linked (deferred) path
    switches itself off per call and the modules run one by one, each inside its unit; ``fused_training=True`` instead keeps the
    projectors in the root unit next to ``feature_fusion`` so the fused forward / backward can read all weights at once.

    Covered: the "3davg" / "avg" resamplers and the un-resampled projectors (with or without ``pre_proj_layernorm``,
    merv.py:165-171) in front of feature_fusion in {cross_attention_avg_lq, scalar, concat_channel, concat_channel_ln} or the
    parameter-free "first" / "concat" (``feature_fusion is None``, merv.py:598-601).
    """
    proj_classes = {"AveragePooling3DProjector": AveragePooling3DProjector, "AveragePoolingProjector": AveragePoolingProjector}
    new_projs = []
    for p in vidlm.projectors:
        name = type(p).__name__
        if name in _PLAIN_PROJECTORS:  # tokens_resampled == False (merv.py:164-172): no pooling, nothing to link
            new_projs.append(_adopt_plain_projector(p))
            fused = False
            continue
        if name == "AttentivePooler":  # "attntv" (merv.py:124-130): its own tokens, nothing to link
            new_projs.append(p if isinstance(p, AttentivePooler) else AttentivePooler.from_reference(p))
            fused = False
            continue
        if name == "Convolutional3DProjector":  # "3dconv" (merv.py:142-150): pooled taps + one GEMM, then the inner projector
            new_projs.append(p if isinstance(p, Convolutional3DProjector) else Convolutional3DProjector.from_reference(p))
            fused = False
            continue
        cls = proj_classes.get(name)
        if cls is None:
            raise TypeError(f"patch_merv supports the 3davg / avg / attntv / 3dconv arch_specifiers and the un-resampled projectors, found {name}")
        new_projs.append(p if isinstance(p, AveragePooling3DProjector) else cls.from_reference(p))
    ff = vidlm.feature_fusion
    fusion_type = getattr(vidlm, "feature_fusion_type", None)
    if ff is None:  # "first" / "concat": glue only (merv.py:598-601)
        new_ff, fused = None, False
    elif type(ff).__name__ == "CrossAttentionAdapterLearnableQuery":
        new_ff = ff if isinstance(ff, CrossAttentionAdapterLearnableQuery) else CrossAttentionAdapterLearnableQuery.from_reference(ff)
    elif type(ff).__name__ == "ScalarAdapter":
        new_ff = ff if isinstance(ff, ScalarAdapter) else ScalarAdapter()
        new_ff.scalar = ff.scalar
    elif type(ff).__name__ == "LinearProjector" and (fusion_type or "concat_channel") == "concat_channel":
        # merv.py:217-218: the glue (merv.py:603-606) concatenates and then calls this module with a tensor -> plain tcgen05 GEMM
        new_ff = ConcatChannelFusion.__new__(ConcatChannelFusion)
        nn.Module.__init__(new_ff)
        new_ff.projector, new_ff.layernorm = ff.projector, ff.layernorm
        new_ff.num_encoder = len(new_projs)
        fused = False
    elif isinstance(ff, nn.Sequential) and len(ff) == 2 and isinstance(ff[0], nn.LayerNorm) and type(ff[1]).__name__ == "LinearProjector":
        # merv.py:219-223 "concat_channel_ln": same two submodules (shared), B200 forward
        new_ff = ConcatChannelLNFusion.__new__(ConcatChannelLNFusion)
        nn.Sequential.__init__(new_ff, ff[0], _adopt_plain_projector(ff[1]))
        new_ff.num_encoder = len(new_projs)
        fused = False
    else:
        raise TypeError("patch_merv supports feature_fusion in {'cross_attention_avg_lq', 'scalar', 'concat_channel', "
                        f"'concat_channel_ln', 'first', 'concat'}}, found {type(ff).__name__}")
    vidlm.projectors = nn.ModuleList(new_projs)
    vidlm.feature_fusion = new_ff
    _extend_fsdp_policy(vidlm, fused_training if fused else None)
    if fused:
        link_fused(new_projs, new_ff)
        if fused_training is not None and isinstance(new_ff, _LinkedMixer):
            new_ff.fused_training = fused_training  # None: per call, fused unless FSDP manages a parameter involved
    return vidlm
