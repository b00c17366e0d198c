"""Training through ``MervFusion.forward_multimodal`` / ``forward_into_embeddings``: the mixer's autograd Function owns the
``[BOS | prefix | text]`` embedding buffer (merv.py:622-720), the kernels write the prefix into its slot and read its gradient from the buffer's
gradient in place, and ``input_embeddings`` get their gradient back through the text rows.

GPU (``-m gpu``): the new strided entry points against their contiguous forms bit for bit (garbage / NaN around the slot), whole training steps
against fp64 autograd through the reference modules plus a torch restatement of merv.py:622-720, bit-identity with ``forward`` + the torch
assembly, the bf16 inference buffer unchanged, no prefix-sized copy in the in-place backward, and determinism.  CPU: the autograd wiring with
the kernels emulated, and the argument checks of the new entry points.  Tolerances (max|a-b| / max|b|): fp32 1e-4, bf16 3e-2.
"""
import ctypes

import pytest
import torch

from oracle import fusion_oracle as O
from oracle.ref_loader import load_reference_nn_utils
from tests import kernel_emulation

DEV = "cuda:0"
TOL = {"fp32": 1e-4, "bf16": 3e-2, "autocast": 3e-2}
OFFSETS = (0.0, 0.5, -0.5, 0.25)
_BT, _L, _K, _EMBED = 5, 6, 128, 48


def _np(t):
    return t.detach().double().cpu().numpy()


def _err(a, b):
    return O.rel_err(_np(a), _np(b))


def _round(t):
    return t.to(torch.bfloat16).to(t.dtype)


# ---- configurations ----------------------------------------------------------------------------------------------------------------------
# frames x S x S pooled tokens per encoder (an encoder in `single` pools to one token); `fused`: the MervFusion fused_training flag
CONFIGS = {
    "lq_fused_t64": dict(mixer="lq", mlp="linear", frames=4, S=4, fused=True),       # T % 128 != 0: prefix computed, then copied into the slot
    "lq_fused_t128": dict(mixer="lq", mlp="linear", frames=8, S=4, fused=True),      # the GEMM stores into the slot
    "lq_module": dict(mixer="lq", mlp="linear", frames=4, S=4, fused=False),
    "lq_gelu": dict(mixer="lq", mlp="gelu-mlp", frames=2, S=2, fused=None),
    "lq_pe": dict(mixer="lq", mlp="linear", frames=2, S=2, fused=None, pe=True),
    "lq_flat": dict(mixer="lq", mlp="linear", frames=2, S=2, fused=None, averagetoken=False),
    "lq_single": dict(mixer="lq", mlp="linear", frames=2, S=2, fused=None, single=(1,)),
    "scalar_fused": dict(mixer="scalar", mlp="linear", frames=4, S=4, fused=True),
    "scalar_gelu": dict(mixer="scalar", mlp="gelu-mlp", frames=2, S=2, fused=None),
    "scalar_fused_t128": dict(mixer="scalar", mlp="linear", frames=8, S=4, fused=True),
}


def _dims(c):
    return (32, 48, 64, 40) if c["mixer"] == "scalar" else (32, 48, 64)


def _setup(cfg, mode, device):
    """(MervFusion, reference projectors, reference mixer, features, text embeddings) on one set of bf16-rounded parameters and inputs."""
    import merv_b200 as M

    ref = load_reference_nn_utils()
    c = CONFIGS[cfg]
    dims, single = _dims(c), c.get("single", ())
    T = c["frames"] * c["S"] ** 2
    torch.manual_seed(11)
    rprojs = [ref.AveragePooling3DProjector(C, _K, 1 if e in single else c["frames"], 1 if e in single else c["S"], mlp_type=c["mlp"])
              for e, C in enumerate(dims)]
    if c["mixer"] == "lq":
        rff = ref.CrossAttentionAdapterLearnableQuery(embed_dim=_EMBED, llm_dim=_K, token_length=T, averagetoken=c.get("averagetoken", True),
                                                      num_encoder=len(dims), positional_embedding=c.get("pe", False))
    else:
        rff = ref.ScalarAdapter(len(dims))
    with torch.no_grad():
        if c["mixer"] == "lq":
            rff.Q.mul_(8.0)  # a mixing softmax far from uniform
            if c.get("pe"):
                rff.pe.mul_(4.0)
        else:
            rff.scalar.copy_(torch.tensor([0.7, -0.4, 0.1, 0.3]))
        for m in rprojs + [rff]:
            for p in m.parameters():
                p.copy_(_round(p))
    projs = [M.AveragePooling3DProjector(C, _K, p.output_frames, p.output_size, c["mlp"]) for C, p in zip(dims, rprojs)]
    for p, r in zip(projs, rprojs):
        p.load_state_dict(r.state_dict())
    if c["mixer"] == "lq":
        ff = M.CrossAttentionAdapterLearnableQuery(_EMBED, _K, T, averagetoken=c.get("averagetoken", True), num_encoder=len(dims),
                                                   positional_embedding=c.get("pe", False))
    else:
        ff = M.ScalarAdapter(len(dims))
    ff.load_state_dict(rff.state_dict())
    m = M.MervFusion(projs, ff, fused_training=c["fused"])
    dtype = torch.bfloat16 if mode == "bf16" else torch.float32
    m = m.to(device=device, dtype=dtype).train()
    g = torch.Generator().manual_seed(3)
    H = 4
    xs = [_round(torch.randn(_BT, 2 * c["frames"], H * H, C, generator=g) + OFFSETS[e]) for e, C in enumerate(dims)]
    emb = _round(torch.randn(_BT, _L, _K, generator=g))
    return m, rprojs, rff, xs, emb, T


def _torch_assemble(prefix, emb, idx, uni, bos):
    """merv.py:622-720 restated with torch.cat / indexing: multimodal rows [BOS | prefix | text], then text-only rows padded at the end."""
    mm = torch.cat([emb[idx, :bos], prefix, emb[idx, bos:]], 1)
    if uni.numel() == 0:
        return mm
    pad = torch.zeros((uni.numel(), prefix.shape[1], emb.shape[2]), dtype=emb.dtype, device=emb.device)
    return torch.cat([mm, torch.cat([emb[uni], pad], 1)], 0)


def _indices(which, device):
    idx = {"all": list(range(_BT)), "two": [3, 0], "one": [4]}[which]
    uni = [i for i in range(_BT) if i not in idx]
    return torch.tensor(idx, device=device), torch.tensor(uni, dtype=torch.long, device=device)


def _loss_tensors(Bm, Bu, T, E, scalar, device):
    g = torch.Generator().manual_seed(5)
    R = torch.randn(Bm + Bu, _L + T, _K, generator=g).to(device)
    r = torch.randn(1 if scalar else Bm, E, generator=g).to(device)
    return R, r


def _step(m, xs, emb, which, bos, mode, device, R=None, r=None):
    """forward_multimodal + backward of loss = sum(R * embeddings) + sum(r * weights); returns (buf, weights, {name: grad}, emb grad)."""
    idx, uni = _indices(which, device)
    dtype = torch.bfloat16 if mode == "bf16" else torch.float32
    m.zero_grad(set_to_none=True)
    e = emb.to(device=device, dtype=dtype).clone().requires_grad_(True)
    feats = [x.to(device=device, dtype=dtype) for x in xs]
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=mode == "autocast"):
        buf, mask, labels, w = m.forward_multimodal(feats, e, multimodal_indices=None if which == "all" else idx, bos_token_length=bos)
    if R is None:
        R, r = _loss_tensors(idx.numel(), uni.numel(), buf.shape[1] - _L, w.shape[1], w.shape[0] == 1 and idx.numel() > 1, device)
    ((buf.float() * R).sum() + (w.float() * r).sum()).backward()
    return buf, w, {k: p.grad for k, p in m.named_parameters()}, e.grad


def _check_against_reference(cfg, mode, which, bos, device):
    m, rprojs, rff, xs, emb, T = _setup(cfg, mode, device)
    buf, w, grads, demb = _step(m, xs, emb, which, bos, mode, device)
    idx, uni = _indices(which, "cpu")
    R, r = _loss_tensors(idx.numel(), uni.numel(), T, w.shape[1], w.shape[0] == 1 and idx.numel() > 1, "cpu")
    rprojs = [p.double() for p in rprojs]
    rff = rff.double()
    e64 = emb.detach().double().requires_grad_(True)
    prefix, want_w = rff([p(x.double()[idx]) for p, x in zip(rprojs, xs)])
    want_buf = _torch_assemble(prefix, e64, idx, uni, bos)
    ((want_buf * R.double()).sum() + (want_w * r.double()).sum()).backward()
    tol = TOL[mode]
    assert buf.shape == want_buf.shape and _err(buf, want_buf) < tol and _err(w, want_w) < tol
    want = {f"projectors.{i}.{k}": p.grad for i, rp in enumerate(rprojs) for k, p in rp.named_parameters()}
    want.update({f"feature_fusion.{k}": p.grad for k, p in rff.named_parameters()})
    assert sorted(grads) == sorted(want)
    for k, ref in want.items():
        got = grads[k]
        if ref is None:  # v_proj_weight / out_proj (dead in the reference too), pe with averagetoken=False
            assert got is None or not got.any(), k
        elif k.endswith("in_proj_bias"):  # b_k / b_v: exactly zero here, rounding noise in the reference
            assert _err(got[:_EMBED], ref[:_EMBED]) < tol and not got[_EMBED:].any(), k
        else:
            assert got is not None and _err(got, ref) < tol, k
    assert demb is not None and _err(demb, e64.grad) < tol
    rest = [i for i in range(_BT) if i not in idx.tolist() + uni.tolist()]
    assert not demb[rest].any()
    return grads


# ---- GPU: the strided entry points against their contiguous forms ------------------------------------------------------------------
def _slot_buffer(B, T, K, dtype, bos=2, L=5, fill=1e4):
    """[B, bos + T + L, K] buffer of large garbage and its prefix slot (rows bos .. bos + T of every video)."""
    g = torch.Generator(device=DEV).manual_seed(T + K)
    buf = (torch.randn(B, bos + T + L, K, generator=g, device=DEV) * fill).to(dtype)
    return buf, buf[:, bos:bos + T]


@pytest.mark.gpu
@pytest.mark.parametrize("T", [64, 128, 192])
def test_wgrad_video_reads_a_batch_strided_slot_bit_identically(T):
    from merv_b200 import _lib, ops

    B, N, C = 3, 256, 192
    g = torch.Generator(device=DEV).manual_seed(T)
    buf, slot = _slot_buffer(B, T, N, torch.bfloat16)
    slot.copy_(torch.randn(B, T, N, generator=g, device=DEV))
    X = torch.randn(B * T, C, generator=g, device=DEV).to(torch.bfloat16)
    W = torch.randn(N, C, generator=g, device=DEV).to(torch.bfloat16)
    scale = torch.rand(B, generator=g, device=DEV) + 0.5
    flat = slot.contiguous().view(B * T, N)
    want_dW, want_p = ops.wgrad_video(flat, X, scale, W, B)
    before = buf.clone()
    dW, p = ops.wgrad_video(slot, X, scale, W, B)
    assert torch.equal(dW, want_dW) and torch.equal(p, want_p) and torch.equal(buf, before)
    # the old entry point is the new one with the packed stride
    lib = _lib.load()
    dW_old, p_old = torch.empty_like(dW), torch.empty_like(p)
    ws = torch.empty(max(int(lib.merv_wgrad_video_workspace(B, N, C)), 4), dtype=torch.float32, device=DEV)
    _lib.check(lib.merv_wgrad_video(flat.data_ptr(), N, X.data_ptr(), C, scale.data_ptr(), 1, W.data_ptr(), C, dW_old.data_ptr(), C,
                                    p_old.data_ptr(), ws.data_ptr(), B, T, N, C, torch.cuda.current_stream().cuda_stream))
    assert torch.equal(dW_old, want_dW) and torch.equal(p_old, want_p)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("mode", ["scores", "weights", "single"])
def test_softmax_mix_ex_writes_the_slot_and_nothing_else(mode, dtype):
    from merv_b200 import _lib, ops

    B, T, K, E = 3, 40, 136 if dtype == torch.float32 else 264, 3
    g = torch.Generator(device=DEV).manual_seed(1)
    Vs = [torch.randn(B, 1 if (mode == "single" and e == 1) else T, K, generator=g, device=DEV).to(dtype) for e in range(E)]
    scores = torch.randn(B, E, generator=g, device=DEV) * 3
    kw = dict(weights=torch.softmax(scores, -1)) if mode == "weights" else dict(scores=scores)
    want, want_w = ops.softmax_mix(Vs, T, **kw)
    buf, slot = _slot_buffer(B, T, K, dtype)
    buf.fill_(float("nan"))
    out, w = ops.softmax_mix(Vs, T, **kw, out=slot)
    assert out.data_ptr() == slot.data_ptr() and torch.equal(slot, want) and torch.equal(w, want_w)
    assert buf[:, :2].isnan().all() and buf[:, 2 + T:].isnan().all()
    # merv_softmax_mix is merv_softmax_mix_ex with the packed strides
    lib = _lib.load()
    old = torch.empty_like(want)
    w_old = torch.empty_like(want_w) if mode != "weights" else kw["weights"]
    _lib.check(lib.merv_softmax_mix(_lib.ptr_array([v.data_ptr() for v in Vs]), _lib.i32_array([v.shape[1] for v in Vs]),
                                    None if mode == "weights" else scores.data_ptr(), w_old.data_ptr(), old.data_ptr(), B, E, T, K,
                                    ops.dtype_code(dtype), torch.cuda.current_stream().cuda_stream))
    assert torch.equal(old, want)


def _mix_case(kind, dtype):
    from merv_b200 import ops

    B, T, K, E, embed = 3, 48, 256, 3, 64
    g = torch.Generator(device=DEV).manual_seed(sum(map(ord, kind)))
    Vs = [torch.randn(B, 1 if (kind == "single" and e == 2) else T, K, generator=g, device=DEV).to(dtype) for e in range(E)]
    per_token_u = kind == "flat"
    Ku = T * K if per_token_u else K
    Q, Wq, Wk, b = ((torch.randn(*s, generator=g, device=DEV) * sc).to(dtype)
                    for s, sc in (((1, embed), 4.0), ((embed, embed), embed ** -0.5), ((embed, Ku), Ku ** -0.5), ((3 * embed,), 0.05)))
    pe = (torch.randn(E, K, generator=g, device=DEV) * 0.1).to(dtype) if kind == "pe" else None
    u = ops.fusion_query_vec(Q, Wq, Wk, b)
    _, weights = ops.softmax_mix(Vs, T, scores=ops.scores_from_tokens(Vs, u, T, per_token_u=per_token_u, mean=not per_token_u))
    dw = torch.randn(B, E, generator=g, device=DEV)
    return Vs, weights, dw, u, Q, Wq, Wk, b, pe, per_token_u, (B, T, K)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["avg", "flat", "single", "pe"])
def test_mix_backward_reads_a_batch_strided_slot_bit_identically(kind, dtype):
    from merv_b200 import ops

    Vs, weights, dw, u, Q, Wq, Wk, b, pe, per_token_u, (B, T, K) = _mix_case(kind, dtype)
    buf, slot = _slot_buffer(B, T, K, dtype)
    slot.copy_(torch.randn(B, T, K, device=DEV))
    want = ops.mix_backward_ex(Vs, slot.contiguous(), weights, dw, u, Q, Wq, Wk, b, per_token_u=per_token_u, pe=pe)
    got = ops.mix_backward_ex(Vs, slot, weights, dw, u, Q, Wq, Wk, b, per_token_u=per_token_u, pe=pe)
    for a, c in zip(want[0], got[0]):
        assert torch.equal(a, c)
    for a, c in zip(want[1:], got[1:]):
        assert (a is None and c is None) or torch.equal(a, c)
    if kind == "avg":
        old = ops.mix_backward(Vs, slot, weights, dw, u, Q, Wq, Wk, b)
        assert all(torch.equal(a, c) for a, c in zip(old[0], want[0])) and all(torch.equal(a, c) for a, c in zip(old[1:], want[1:5]))
    _check_old_mix_backward_ex(Vs, slot.contiguous(), weights, dw, u, Q, Wq, Wk, b, pe, per_token_u, want)


def _check_old_mix_backward_ex(Vs, dout, weights, dw, u, Q, Wq, Wk, b, pe, per_token_u, want):
    """merv_mix_backward_ex called directly (it is merv_mix_backward_strided with the packed strides): the same bits."""
    from merv_b200 import _lib, ops

    lib = _lib.load()
    B, T, K = dout.shape
    E, embed, dt = len(Vs), Wk.shape[0], dout.dtype
    dVs = [torch.empty_like(v) for v in Vs]
    dQ, dWq, dWk, dbias = (torch.empty(s, dtype=dt, device=DEV) for s in ((1, embed), (embed, embed), tuple(Wk.shape), (3 * embed,)))
    dpe = None if pe is None else torch.empty_like(pe)
    n = lib.merv_mix_backward_ex_workspace(B, E, T, K, embed, K if per_token_u else 0)
    ws = torch.empty(n, dtype=torch.float32, device=DEV)
    _lib.check(lib.merv_mix_backward_ex(_lib.ptr_array([v.data_ptr() for v in Vs]), _lib.i32_array([v.shape[1] for v in Vs]), dout.data_ptr(),
                                        weights.data_ptr(), dw.data_ptr(), u.data_ptr(), K if per_token_u else 0, None if pe is None else pe.data_ptr(),
                                        0 if pe is None else pe.stride(0), Q.data_ptr(), Wq.data_ptr(), Wk.data_ptr(), b.data_ptr(),
                                        _lib.ptr_array([d.data_ptr() for d in dVs]), dQ.data_ptr(), dWq.data_ptr(), dWk.data_ptr(), dbias.data_ptr(),
                                        None if dpe is None else dpe.data_ptr(), ws.data_ptr(), n, B, E, T, K, embed, ops.dtype_code(dt),
                                        torch.cuda.current_stream().cuda_stream))
    assert all(torch.equal(a, c) for a, c in zip(dVs, want[0]))
    assert all(torch.equal(a, c) for a, c in zip((dQ, dWq, dWk, dbias), want[1:5]))
    assert dpe is None or torch.equal(dpe, want[5])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_scalar_mix_backward_reads_a_batch_strided_slot_bit_identically(dtype):
    from merv_b200 import _lib, ops

    B, T, K, E = 3, 37, 264, 4
    g = torch.Generator(device=DEV).manual_seed(9)
    Vs = [torch.randn(B, T, K, generator=g, device=DEV).to(dtype) for _ in range(E)]
    w = torch.softmax(torch.randn(E, generator=g, device=DEV), 0)
    dw = torch.randn(E, generator=g, device=DEV)
    buf, slot = _slot_buffer(B, T, K, dtype)
    slot.copy_(torch.randn(B, T, K, generator=g, device=DEV))
    want_dV, want_ds = ops.scalar_mix_backward(Vs, slot.contiguous(), w, dw)
    dV, ds = ops.scalar_mix_backward(Vs, slot, w, dw)
    assert all(torch.equal(a, c) for a, c in zip(dV, want_dV)) and torch.equal(ds, want_ds)
    lib = _lib.load()
    dV_old, ds_old = [torch.empty_like(v) for v in Vs], torch.empty_like(ds)
    n = lib.merv_scalar_mix_backward_workspace(B, E, K)
    ws = torch.empty(n, dtype=torch.float32, device=DEV)
    flat = slot.contiguous()
    _lib.check(lib.merv_scalar_mix_backward(_lib.ptr_array([v.data_ptr() for v in Vs]), flat.data_ptr(), w.data_ptr(), dw.data_ptr(),
                                            _lib.ptr_array([d.data_ptr() for d in dV_old]), ds_old.data_ptr(), ws.data_ptr(), n, B, E, T, K,
                                            ops.dtype_code(dtype), torch.cuda.current_stream().cuda_stream))
    assert all(torch.equal(a, c) for a, c in zip(dV_old, want_dV)) and torch.equal(ds_old, want_ds)


# ---- GPU: whole training steps -----------------------------------------------------------------------------------------------------
STEP_CASES = [(cfg, mode) for cfg in CONFIGS for mode in ("fp32", "autocast", "bf16")
              if not (CONFIGS[cfg]["fused"] and mode == "fp32")]  # the fused step is bf16 only (fp32 trains module by module)


@pytest.mark.gpu
@pytest.mark.parametrize("which,bos", [("all", 1), ("two", 2), ("one", 1)])
@pytest.mark.parametrize("cfg,mode", STEP_CASES)
def test_forward_multimodal_training_matches_reference(cfg, mode, which, bos):
    _check_against_reference(cfg, mode, which, bos, DEV)


def _expected_fn(cfg, mode):
    c = CONFIGS[cfg]
    if c["fused"] and mode != "fp32":
        return "_FusedLinearFn" if c["mixer"] == "lq" else "_FusedScalarLinearFn"
    return "_MixFn" if c["mixer"] == "lq" else "_ScalarMixFn"


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["lq_fused_t64", "lq_fused_t128", "lq_module", "lq_single", "scalar_fused", "scalar_gelu"])
def test_gradients_equal_forward_plus_torch_assembly_bit_for_bit(cfg):
    """The kernels do the same reductions whether dOut is the slot of the buffer's gradient or the narrow view the concat's backward gives."""
    import merv_b200 as M  # noqa: F401

    m, _, _, xs, emb, T = _setup(cfg, "bf16", DEV)
    idx, uni = _indices("two", DEV)
    bos = 2
    buf, w, grads, demb = _step(m, xs, emb, "two", bos, "bf16", DEV)
    assert type(buf.grad_fn).__name__.startswith(_expected_fn(cfg, "bf16"))
    R, r = _loss_tensors(idx.numel(), uni.numel(), T, w.shape[1], CONFIGS[cfg]["mixer"] == "scalar", DEV)
    m.zero_grad(set_to_none=True)
    e = emb.to(DEV, torch.bfloat16).requires_grad_(True)
    prefix, w2 = m([x.to(DEV, torch.bfloat16).index_select(0, idx) for x in xs])
    buf2 = _torch_assemble(prefix, e, idx, uni, bos)
    ((buf2.float() * R).sum() + (w2.float() * r).sum()).backward()
    assert torch.equal(buf, buf2) and torch.equal(w, w2)
    for k, g in grads.items():
        p = dict(m.named_parameters())[k]
        assert (g is None and p.grad is None) or torch.equal(g, p.grad), k
    assert torch.equal(demb, e.grad)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["lq_fused_t128"])
def test_training_buffer_equals_the_inference_buffer(cfg):
    m, _, _, xs, emb, T = _setup(cfg, "bf16", DEV)
    idx, _ = _indices("two", DEV)
    feats = [x.to(DEV, torch.bfloat16) for x in xs]
    e = emb.to(DEV, torch.bfloat16)
    with torch.no_grad():
        want, _, _, want_w = m.forward_multimodal(feats, e, multimodal_indices=idx, bos_token_length=2)
    buf, _, _, w = m.forward_multimodal(feats, e, multimodal_indices=idx, bos_token_length=2)
    assert type(buf.grad_fn).__name__.startswith("_FusedLinearFn")
    assert torch.equal(buf, want) and torch.equal(w, want_w)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["lq_fused_t128", "scalar_fused_t128"])
def test_in_place_backward_copies_no_prefix(cfg):
    """T % 128 == 0: no copy / clone / contiguous of a prefix-sized tensor in the fused backward."""
    from torch.profiler import ProfilerActivity, profile

    m, _, _, xs, emb, T = _setup(cfg, "bf16", DEV)
    idx, _ = _indices("two", DEV)
    e = emb.to(DEV, torch.bfloat16).requires_grad_(True)
    buf, _, _, w = m.forward_multimodal([x.to(DEV, torch.bfloat16) for x in xs], e, multimodal_indices=idx, bos_token_length=1)
    R = torch.randn(buf.shape, device=DEV).to(buf.dtype)  # in the buffer's dtype: the loss itself converts nothing
    loss = (buf * R).sum() + w.float().sum()
    with profile(activities=[ProfilerActivity.CPU], record_shapes=True) as prof:
        loss.backward()
    limit = idx.numel() * T * _K
    big = []
    for ev in prof.events():
        if ev.name in ("aten::copy_", "aten::clone", "aten::contiguous"):
            for shape in ev.input_shapes:
                n = 1
                for s in shape or []:
                    n *= s
                if shape and n >= limit:
                    big.append((ev.name, shape))
    assert not big, big
    assert e.grad is not None


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["lq_fused_t128", "lq_module", "scalar_fused"])
def test_two_training_steps_are_bit_identical(cfg):
    m, _, _, xs, emb, _ = _setup(cfg, "bf16", DEV)
    _, _, first, d1 = _step(m, xs, emb, "two", 1, "bf16", DEV)
    first = {k: None if g is None else g.clone() for k, g in first.items()}
    _, _, second, d2 = _step(m, xs, emb, "two", 1, "bf16", DEV)
    for k in first:
        assert (first[k] is None and second[k] is None) or torch.equal(first[k], second[k]), k
    assert torch.equal(d1, d2)


# ---- CPU: the autograd wiring with the kernels emulated --------------------------------------------------------------------------------
def _emulate(monkeypatch):
    """kernel_emulation plus the new arguments: ``out=`` of softmax_mix, a [videos, T, N] dY of wgrad_video, and the mix backwards."""
    from merv_b200 import ops
    from tests.test_adapter_backward_variants import _mix_backward_ex_standin
    from tests.test_scalar_adapter_training import _scalar_fused_backward_standin, _scalar_mix_backward_standin

    kernel_emulation.emulate(monkeypatch)
    calls = []

    def softmax_mix(Vs, token_length, scores=None, weights=None, out=None):
        res, w = kernel_emulation.softmax_mix(Vs, token_length, scores=scores, weights=weights)
        if out is None:
            return res, w
        calls.append("softmax_mix_out")
        out.copy_(res)
        return out, w

    def wgrad_video(dy, x, scale, w, videos):
        if dy.dim() == 3:
            calls.append("wgrad_strided" if not dy.is_contiguous() else "wgrad_3d")
            dy = dy.reshape(-1, dy.shape[2])
        return kernel_emulation.wgrad_video(dy, x, scale, w, videos)

    def mix_backward(Vs, dout, weights, dweights, u, Q, Wq, Wk, b):
        calls.append("mix_backward" + ("" if dout.is_contiguous() else "_strided"))
        return _mix_backward_ex_standin(Vs, dout, weights, dweights, u, Q, Wq, Wk, b)[:5]

    def scalar_mix_backward(Vs, dout, weights, dweights=None):
        calls.append("scalar_mix_backward" + ("" if dout.is_contiguous() else "_strided"))
        return _scalar_mix_backward_standin(Vs, dout, weights, dweights)

    monkeypatch.setattr(ops, "softmax_mix", softmax_mix)
    monkeypatch.setattr(ops, "wgrad_video", wgrad_video)
    monkeypatch.setattr(ops, "mix_backward", mix_backward)
    monkeypatch.setattr(ops, "mix_backward_ex", _mix_backward_ex_standin)
    monkeypatch.setattr(ops, "scalar_mix_backward", scalar_mix_backward)
    monkeypatch.setattr(ops, "scalar_fused_backward", _scalar_fused_backward_standin)
    return calls


@pytest.mark.parametrize("which,bos", [("two", 2), ("one", 1)])
@pytest.mark.parametrize("cfg,mode", [("lq_module", "fp32"), ("lq_fused_t128", "bf16"), ("lq_fused_t64", "bf16"), ("scalar_gelu", "fp32"),
                                      ("scalar_fused", "bf16")])
def test_wiring_matches_reference_on_cpu(cfg, mode, which, bos, monkeypatch):
    """The module code unchanged, the kernels emulated: the buffer is spliced as merv.py:622-720 does, the prefix gradient is handed to the
    kernels as the slot of the buffer's gradient, and input_embeddings get the text gradients back (zeros in rows outside both index sets)."""
    calls = _emulate(monkeypatch)
    _check_against_reference(cfg, mode, which, bos, "cpu")
    fused = CONFIGS[cfg]["fused"] and mode == "bf16"
    strided = which != "one"  # the slot of a single video is a contiguous tensor
    if fused:
        assert ("wgrad_strided" in calls) == strided
    else:
        assert "softmax_mix_out" in calls and any(c.endswith("_strided") for c in calls) == strided


def test_input_embeddings_get_a_gradient_only_when_they_require_one(monkeypatch):
    _emulate(monkeypatch)
    m, _, _, xs, emb, T = _setup("lq_module", "fp32", "cpu")
    idx = torch.tensor([3, 0])
    buf, w = m.forward_into_embeddings(xs, emb, bos_token_length=1, multimodal_indices=idx)
    assert buf.shape == (2, _L + T, _K) and torch.equal(buf[:, :1], emb[idx, :1]) and torch.equal(buf[:, 1 + T:], emb[idx, 1:])
    buf.sum().backward()
    assert emb.grad is None and m.feature_fusion.Q.grad is not None
    m.zero_grad(set_to_none=True)
    e = emb.clone().requires_grad_(True)
    buf, w = m.forward_into_embeddings(xs, e, bos_token_length=1, multimodal_indices=idx)
    buf.sum().backward()
    want = torch.zeros_like(emb)
    want[idx] = 1.0
    assert torch.equal(e.grad, want)


def test_unimodal_rows_are_padded_with_zeros_on_cpu(monkeypatch):
    _emulate(monkeypatch)
    m, _, _, xs, emb, T = _setup("scalar_gelu", "fp32", "cpu")
    mask, labels = torch.ones(_BT, _L, dtype=torch.bool), torch.arange(_BT * _L).reshape(_BT, _L)
    buf, fm, fl, w = m.forward_multimodal(xs, emb, mask, labels, multimodal_indices=torch.tensor([4]), bos_token_length=1)
    assert buf.shape == (_BT, _L + T, _K) and w.shape == (1, 4)
    assert torch.equal(buf[1:, :_L], emb[:4]) and not buf[1:, _L:].any()
    assert fm[0].all() and not fm[1:, _L:].any() and (fl[0, 1:1 + T] == -100).all()


# ---- CPU: argument checks of the new entry points ----------------------------------------------------------------------------------
def test_new_entry_points_argument_checks():
    """Checks that run before any device is touched: NULL pointers, strides that are not whole 16-byte vectors, batch strides that would
    make two videos overlap."""
    from merv_b200 import _lib

    lib = _lib.load()
    B, T, K, E, embed = 2, 64, 128, 3, 32
    fake = ctypes.c_void_p(256)
    ptrs = _lib.ptr_array([256] * 8)
    tokens = _lib.i32_array([T] * E)
    err = lib.merv_last_error

    def wgrad(dY=fake, lddy=K, bs=(T + 3) * K):
        return lib.merv_wgrad_video_ex(dY, lddy, bs, fake, 64, fake, 1, fake, 64, fake, 64, fake, fake, B, T, K, 64, None)

    assert wgrad(dY=None) == -6 and b"NULL" in err()
    assert wgrad(lddy=K + 4) == -2 and wgrad(bs=(T + 3) * K + 4) == -2 and b"multiple" in err()
    assert wgrad(dY=ctypes.c_void_p(264)) == -2
    assert wgrad(bs=T * K - 8) == -1 and b"overlap" in err()

    def mix(out=fake, ldo=K, bs=(T + 3) * K, dtype=_lib.MERV_BF16):
        return lib.merv_softmax_mix_ex(ptrs, tokens, fake, fake, out, ldo, bs, B, E, T, K, dtype, None)

    assert mix(out=None) == -6 and b"NULL" in err()
    assert mix(ldo=K + 4) == -2 and mix(bs=(T + 3) * K + 4) == -2 and b"16-byte" in err()
    assert mix(ldo=K + 4, dtype=_lib.MERV_F32) != -2  # 4 fp32 elements are one 16-byte vector
    assert mix(bs=T * K - 8) == -1 and b"overlap" in err()
    assert mix(ldo=K - 8) == -1

    def mixb(dOut=fake, ldo=K, bs=(T + 3) * K):
        return lib.merv_mix_backward_strided(ptrs, tokens, dOut, ldo, bs, fake, None, fake, 0, None, 0, fake, fake, fake, fake, ptrs, fake, fake,
                                             fake, fake, None, fake, 1 << 20, B, E, T, K, embed, _lib.MERV_BF16, None)

    assert mixb(dOut=None) == -6 and b"NULL" in err()
    assert mixb(ldo=K + 4) == -2 and mixb(bs=(T + 3) * K + 4) == -2 and mixb(dOut=ctypes.c_void_p(264)) == -2
    assert mixb(bs=T * K - 8) == -1 and b"overlap" in err()

    n = lib.merv_scalar_mix_backward_workspace(B, 4, K)

    def scal(dOut=fake, ldo=K, bs=(T + 3) * K):
        return lib.merv_scalar_mix_backward_strided(ptrs, dOut, ldo, bs, fake, None, ptrs, fake, fake, n, B, 4, T, K, _lib.MERV_BF16, None)

    assert scal(dOut=None) == -6 and b"NULL" in err()
    assert scal(ldo=K + 4) == -2 and scal(bs=(T + 3) * K + 4) == -2 and scal(dOut=ctypes.c_void_p(264)) == -2
    assert scal(bs=T * K - 8) == -1 and b"overlap" in err()
