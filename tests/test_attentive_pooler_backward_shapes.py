"""Training the attentive pooler (``attntv``, AttentivePooler) at every shape and dtype its forward runs.

The attention backward has two kernels behind ``merv_cross_attention_backward_ex``: the tcgen05 one for bf16 frames inside its tile
(n_q <= 64, n_kv <= 256, head_dim % 32 == 0) and a CUDA-core one for everything else (any n_q / n_kv, head_dim <= 128 and a multiple
of 8 in bf16 / 4 in fp32, fp32 and bf16).  ``MERV_ATTN_IMPL=simt`` forces the CUDA-core kernel.

GPU (``-m gpu``): ``ops.cross_attention_backward`` against fp64 autograd on the same rounded inputs, dQ / dK / dV checked separately as
``max|a-b| <= tol * max|ref|`` (fp32 1e-5, bf16 CUDA cores 1e-2, bf16 tcgen05 1.5e-2), over the tails of the 64-key chunks and the
64-query blocks, shared and per-entry queries and padded rows; bit-reproducibility and frame-alone == frame-in-batch; the tcgen05
branch of ``_ex`` bit-identical to ``merv_cross_attention_backward``, whose domain is unchanged; and whole training steps of the module
and of ``MervFusion`` (``attntv+linear``) against the reference modules.  CPU: the fp32 autograd wiring with the kernels emulated, and
the argument checks of the new entry points.
"""
import copy
import ctypes

import pytest
import torch

from oracle import fusion_oracle as O
from oracle.ref_loader import load_reference_nn_utils
from tests import kernel_emulation

DEV = "cuda:0"
FP32_TOL = 1e-5
SIMT_BF16_TOL = 1e-2
TC_TOL = 1.5e-2


# ---- kernel level ------------------------------------------------------------------------------------------------------------------
def _inputs(dtype, batches, n_q, n_kv, heads, hd, shared_q=True, pad=0, seed=0, peaked=False, equal=False):
    """q [n_q, C] or [batches, n_q, C], kv [batches * n_kv, 2C], dout [batches, n_q, C] on the GPU in `dtype`; pad > 0 gives q and kv rows
    `pad` elements longer than their data (strided views)."""
    g = torch.Generator().manual_seed(seed)
    C_ = heads * hd
    q = torch.randn((n_q, C_ + pad) if shared_q else (batches, n_q, C_ + pad), generator=g)
    kv = torch.randn((batches * n_kv, 2 * C_ + pad), generator=g)
    dout = torch.randn((batches, n_q, C_), generator=g)
    if peaked:  # one dominant key per frame and head: the softmax is nearly one-hot
        q = q * 20.0
        kv.view(batches, n_kv, -1)[:, n_kv // 2, :C_] = q.reshape(-1, n_q, C_ + pad)[0, 0, :C_] / 20.0
    if equal:  # every score equal, so the softmax is uniform: the queries live in the first half of each head's dims, where every key is 1
        first = (torch.arange(C_) % hd) < hd // 2
        q[..., :C_][..., ~first] = 0.0
        kv[:, :C_][:, first] = 1.0
    q = q.to(dtype).to(DEV)[..., :C_]
    kv = kv.to(dtype).to(DEV)[:, :2 * C_]
    return q, kv, dout.to(dtype).to(DEV)


def _reference(q, kv, dout, batches, heads):
    """fp64 autograd through the attention of CrossAttention.forward (nn_utils.py:393-412) on the inputs as the kernel received them."""
    C_ = q.shape[-1]
    n_q, hd = q.shape[-2], C_ // heads
    n_kv = kv.shape[0] // batches
    qq = (q.double().unsqueeze(0).expand(batches, n_q, C_) if q.dim() == 2 else q.double()).clone().requires_grad_(True)
    kk = kv.double().clone().requires_grad_(True)
    k5 = kk.view(batches, n_kv, 2, heads, hd)
    qh = qq.view(batches, n_q, heads, hd).permute(0, 2, 1, 3)
    att = torch.softmax(qh @ k5[:, :, 0].permute(0, 2, 3, 1) * hd ** -0.5, -1)
    out = (att @ k5[:, :, 1].permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(batches, n_q, C_)
    return torch.autograd.grad(out, [qq, kk], dout.double())


def _check(got, want, C_, tol):
    dq, dkv = got
    want_dq, want_dkv = want
    for name, a, b in (("dQ", dq, want_dq), ("dK", dkv[:, :C_], want_dkv[:, :C_]), ("dV", dkv[:, C_:], want_dkv[:, C_:])):
        assert a.shape == b.shape, name
        err, scale = float((a.double() - b).abs().max()), float(b.abs().max())
        assert err <= tol * scale, f"{name}: max|err| / max|ref| = {err / max(scale, 1e-300):.3e} > {tol:.1e}"


def _run_simt(monkeypatch, dtype, batches, n_q, n_kv, heads, hd, **kw):
    from merv_b200 import ops

    monkeypatch.setenv("MERV_ATTN_IMPL", "simt")
    q, kv, dout = _inputs(dtype, batches, n_q, n_kv, heads, hd, **kw)
    got = ops.cross_attention_backward(q, kv, dout, batches, heads)
    assert got[0].dtype == dtype and got[1].dtype == dtype
    _check(got, _reference(q, kv, dout, batches, heads), heads * hd, FP32_TOL if dtype == torch.float32 else SIMT_BF16_TOL)
    return q, kv, dout, got


DTYPES = pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])


@pytest.mark.gpu
@DTYPES
@pytest.mark.parametrize("n_kv", [1, 9, 64, 65, 196, 257, 729])
@pytest.mark.parametrize("n_q", [1, 5, 64, 65, 128, 144, 256])
def test_simt_backward_matches_fp64_over_chunk_and_block_tails(monkeypatch, dtype, n_q, n_kv):
    _run_simt(monkeypatch, dtype, 3, n_q, n_kv, 2, 40, seed=n_q * 1000 + n_kv)


@pytest.mark.gpu
@DTYPES
@pytest.mark.parametrize("n_q,n_kv", [(144, 65), (5, 729)])
@pytest.mark.parametrize("hd", [4, 8, 40, 96, 128])
def test_simt_backward_matches_fp64_at_every_head_dim(monkeypatch, dtype, hd, n_q, n_kv):
    if hd == 4 and dtype == torch.bfloat16:
        pytest.skip("bf16 head_dim is a multiple of 8")
    _run_simt(monkeypatch, dtype, 2, n_q, n_kv, 3, hd, seed=hd)


@pytest.mark.gpu
@DTYPES
@pytest.mark.parametrize("pad", [0, 8], ids=["dense", "padded"])
@pytest.mark.parametrize("shared_q", [True, False], ids=["shared", "per_entry"])
def test_simt_backward_query_layouts_and_row_strides(monkeypatch, dtype, shared_q, pad):
    _, _, _, (dq, dkv) = _run_simt(monkeypatch, dtype, 4, 65, 257, 2, 40, shared_q=shared_q, pad=pad, seed=7)
    assert dq.shape == (4, 65, 80) and dkv.shape == (4 * 257, 160)


@pytest.mark.gpu
@DTYPES
@pytest.mark.parametrize("mode", ["peaked", "equal"])
def test_simt_backward_peaked_and_uniform_softmax(monkeypatch, dtype, mode):
    _run_simt(monkeypatch, dtype, 2, 70, 200, 2, 40, seed=3, peaked=mode == "peaked", equal=mode == "equal")


@pytest.mark.gpu
@DTYPES
@pytest.mark.parametrize("shared_q", [True, False], ids=["shared", "per_entry"])
def test_simt_backward_is_bit_reproducible_and_frame_independent(monkeypatch, dtype, shared_q):
    from merv_b200 import ops

    monkeypatch.setenv("MERV_ATTN_IMPL", "simt")
    B, n_q, n_kv, heads = 40, 65, 130, 2
    q, kv, dout = _inputs(dtype, B, n_q, n_kv, heads, 40, shared_q=shared_q, seed=11)
    dq, dkv = ops.cross_attention_backward(q, kv, dout, B, heads)
    dq2, dkv2 = ops.cross_attention_backward(q, kv, dout, B, heads)
    assert torch.equal(dq, dq2) and torch.equal(dkv, dkv2)
    for b in (0, 17, 39):
        qb = q if shared_q else q[b:b + 1]
        dq1, dkv1 = ops.cross_attention_backward(qb, kv[b * n_kv:(b + 1) * n_kv], dout[b:b + 1], 1, heads)
        assert torch.equal(dq1[0], dq[b]) and torch.equal(dkv1, dkv[b * n_kv:(b + 1) * n_kv]), b


TC_SHAPES = [(8, 128, 64, 256, 3, True), (8, 96, 64, 196, 2, True), (2, 32, 37, 70, 1, True), (3, 64, 64, 200, 5, False)]


def _old_entry(q, kv, dout, batches, heads):
    """merv_cross_attention_backward called directly: (rc, dq, dkv)."""
    from merv_b200 import _lib

    lib = _lib.load()
    C_ = q.shape[-1]
    n_q, n_kv, hd = q.shape[-2], kv.shape[0] // batches, C_ // heads
    dq = torch.full((batches, n_q, C_), float("nan"), dtype=q.dtype, device=DEV)
    dkv = torch.full((batches * n_kv, 2 * C_), float("nan"), dtype=q.dtype, device=DEV)
    rc = lib.merv_cross_attention_backward(q.data_ptr(), q.stride(-2), 0 if q.dim() == 2 else q.stride(0), kv.data_ptr(), kv.stride(0),
                                           dout.data_ptr(), dout.stride(1), dq.data_ptr(), dq.stride(1), dkv.data_ptr(), dkv.stride(0), batches,
                                           n_q, n_kv, heads, hd, float(hd ** -0.5), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, dq, dkv


@pytest.mark.gpu
@pytest.mark.parametrize("heads,hd,n_q,n_kv,batches,shared_q", TC_SHAPES)
def test_tcgen05_shapes_both_kernels_meet_their_bounds_and_ex_matches_the_old_entry(monkeypatch, heads, hd, n_q, n_kv, batches, shared_q):
    from merv_b200 import _lib, ops

    lib = _lib.load()
    q, kv, dout = _inputs(torch.bfloat16, batches, n_q, n_kv, heads, hd, shared_q=shared_q, seed=hd + n_kv)
    want = _reference(q, kv, dout, batches, heads)
    assert lib.merv_cross_attention_backward_ex_workspace(batches, n_q, n_kv, heads, hd, _lib.MERV_BF16) == 0  # the tcgen05 kernel runs
    tc = ops.cross_attention_backward(q, kv, dout, batches, heads)
    _check(tc, want, heads * hd, TC_TOL)
    rc, dq_old, dkv_old = _old_entry(q, kv, dout, batches, heads)
    assert rc == 0 and torch.equal(tc[0], dq_old) and torch.equal(tc[1], dkv_old)
    monkeypatch.setenv("MERV_ATTN_IMPL", "simt")
    assert lib.merv_cross_attention_backward_ex_workspace(batches, n_q, n_kv, heads, hd, _lib.MERV_BF16) > 0
    simt = ops.cross_attention_backward(q, kv, dout, batches, heads)
    _check(simt, want, heads * hd, SIMT_BF16_TOL)
    rc, dq_old2, dkv_old2 = _old_entry(q, kv, dout, batches, heads)  # the old entry point has no workspace: always the tcgen05 kernel
    assert rc == 0 and torch.equal(dq_old2, dq_old) and torch.equal(dkv_old2, dkv_old)


@pytest.mark.gpu
@pytest.mark.parametrize("n_q,n_kv,hd", [(65, 64, 32), (64, 257, 32), (64, 64, 40), (144, 729, 128)])
def test_old_entry_point_still_rejects_shapes_outside_the_tcgen05_tile(n_q, n_kv, hd):
    from merv_b200 import _lib

    q, kv, dout = _inputs(torch.bfloat16, 1, n_q, n_kv, 2, hd)
    rc, _, _ = _old_entry(q, kv, dout, 1, 2)
    assert rc == -1 and b"at most" in _lib.load().merv_last_error()  # MERV_E_SHAPE from the tcgen05 kernel's own check


# ---- module level ------------------------------------------------------------------------------------------------------------------
def _perturbed_reference(C_, llm, n, heads, F, mlp_type, seed):
    ref = load_reference_nn_utils()
    torch.manual_seed(seed)
    r = ref.AttentivePooler(C_, llm, num_query_tokens=n, num_heads=heads, output_frames=F, mlp_type=mlp_type)
    with torch.no_grad():  # non-trivial biases / norms / queries (zeros / ones / std 0.02 by default)
        for name, p in r.named_parameters():
            if name.endswith("bias") or "norm" in name:
                p.add_(0.1 * torch.randn_like(p))
        r.query_tokens.mul_(20.0)
    return r


def _grads_within(m, r, rel):
    got = dict(m.named_parameters())
    seen = 0
    for name, p in r.named_parameters():
        assert got[name].grad is not None, name
        scale = float(p.grad.abs().max())
        err = float((got[name].grad.double() - p.grad.double()).abs().max())
        assert err <= rel * scale + 1e-12, (name, err / max(scale, 1e-300))
        seen += 1
    return seen


@pytest.mark.gpu
@pytest.mark.parametrize("C_,llm,n,heads,F,N,B,mlp_type", [(64, 48, 8, 2, 3, 9, 2, "gelu-mlp"), (256, 128, 144, 8, 2, 196, 1, "gelu-mlp"),
                                                          (320, 128, 64, 8, 2, 729, 1, "linear")])
def test_attentive_pooler_fp32_training_matches_fp64_reference(monkeypatch, C_, llm, n, heads, F, N, B, mlp_type):
    import merv_b200 as M

    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    r = _perturbed_reference(C_, llm, n, heads, F, mlp_type, C_ + n)
    m = M.AttentivePooler.from_reference(copy.deepcopy(r)).to(DEV)
    r = r.double().to(DEV)
    g = torch.Generator().manual_seed(5)
    x = torch.randn((B, F, N, C_), generator=g).to(DEV)
    G = torch.randn((B, F * n, llm), generator=g).to(DEV)
    out = m(x)
    assert out.dtype == torch.float32 and out.requires_grad
    out.backward(G)
    want = r(x.double())
    want.backward(G.double())
    torch.cuda.synchronize()
    assert O.rel_err(out.detach().double().cpu().numpy(), want.detach().cpu().numpy()) < 1e-5
    assert _grads_within(m, r, 1e-4) == (19 if mlp_type == "gelu-mlp" else 17)


@pytest.mark.gpu
def test_attentive_pooler_bf16_training_outside_the_tcgen05_tile_matches_reference():
    """n_q 144 and n_kv 729 with head_dim 40: every attention backward of this step runs on the CUDA cores."""
    import merv_b200 as M

    C_, llm, n, heads, F, N, B = 320, 128, 144, 8, 2, 729, 1
    r = _perturbed_reference(C_, llm, n, heads, F, "gelu-mlp", 9)
    m = M.AttentivePooler.from_reference(copy.deepcopy(r)).to(device=DEV, dtype=torch.bfloat16)
    r = r.to(torch.bfloat16).float().to(DEV)
    g = torch.Generator().manual_seed(5)
    x = torch.randn((B, F, N, C_), generator=g).to(torch.bfloat16).to(DEV)
    G = torch.randn((B, F * n, llm), generator=g).to(DEV)
    out = m(x)
    out.backward(G.to(torch.bfloat16))
    want = r(x.float())
    want.backward(G)
    torch.cuda.synchronize()
    assert O.rel_err(out.detach().float().cpu().numpy(), want.detach().cpu().numpy()) < 2e-2
    assert _grads_within(m, r, 4e-2) == 19


_DIMS, _LLM, _TEMPORAL, _PTL, _N = [64, 128], 64, [2, 2], 144, [49, 16]


def _fusion_and_reference():
    """MervFusion('attntv+linear', learnable-query adapter, 144 query tokens per frame) and the reference modules built in
    MERV.__init__'s order (merv.py:87-227) from the same seed."""
    import merv_b200 as M

    vfl = _TEMPORAL[0] * _PTL
    m = M.MervFusion.from_config(_DIMS, _LLM, _TEMPORAL, arch_specifier="attntv+linear", feature_fusion="cross_attention_avg_lq",
                                 projector_token_length=_PTL, visual_feature_length=vfl)
    ref = load_reference_nn_utils()
    torch.manual_seed(_DIMS[0])
    projs = [ref.AttentivePooler(c, _LLM, num_query_tokens=_PTL, num_heads=8, output_frames=t, mlp_type="linear") for c, t in zip(_DIMS, _TEMPORAL)]
    ff = ref.CrossAttentionAdapterLearnableQuery(embed_dim=3072, llm_dim=_LLM, token_length=vfl, averagetoken=True)
    want_sd = {f"projectors.{k}": v for k, v in torch.nn.ModuleList(projs).state_dict().items()}
    want_sd.update({f"feature_fusion.{k}": v for k, v in ff.state_dict().items()})
    got_sd = m.state_dict()
    assert list(got_sd) == list(want_sd) and all(torch.equal(got_sd[k], want_sd[k]) for k in want_sd)
    return m, projs, ff


@pytest.mark.gpu
@pytest.mark.parametrize("autocast", [False, True], ids=["fp32", "bf16_autocast"])
def test_merv_fusion_attntv_training_step_matches_reference(monkeypatch, autocast):
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    m, projs, ff = _fusion_and_reference()
    m = m.to(DEV).train()
    g = torch.Generator().manual_seed(3)
    xs = [torch.randn(1, t, N, c, generator=g) for c, t, N in zip(_DIMS, _TEMPORAL, _N)]
    if autocast:  # the same bf16-rounded features on both sides
        xs = [x.to(torch.bfloat16).float() for x in xs]
    G = torch.randn(1, _TEMPORAL[0] * _PTL, _LLM, generator=g)
    H = torch.randn(1, len(_DIMS), generator=g)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        out, w = m([x.to(DEV) for x in xs])
        ((out.float() * G.to(DEV)).sum() + (w.float() * H.to(DEV)).sum()).backward()
    rdt = torch.float32 if autocast else torch.float64
    projs = [p.to(device=DEV, dtype=rdt) for p in projs]
    ff = ff.to(device=DEV, dtype=rdt)
    want_out, want_w = ff([p(x.to(device=DEV, dtype=rdt)) for p, x in zip(projs, xs)])
    ((want_out * G.to(DEV, rdt)).sum() + (want_w * H.to(DEV, rdt)).sum()).backward()
    torch.cuda.synchronize()
    tol, gtol = (2e-2, 4e-2) if autocast else (1e-5, 1e-4)
    assert O.rel_err(out.detach().double().cpu().numpy(), want_out.detach().double().cpu().numpy()) < tol
    want = {f"projectors.{i}.{k}": p.grad for i, r in enumerate(projs) for k, p in r.named_parameters()}
    want.update({f"feature_fusion.{k}": p.grad for k, p in ff.named_parameters()})
    for k, p in m.named_parameters():
        rg = want[k]
        if rg is None:  # parameters the reference's forward never reads (the adapter's v / out projections)
            assert p.grad is None or not p.grad.any(), k
            continue
        assert p.grad is not None, k
        scale = float(rg.abs().max())
        err = float((p.grad.double() - rg.double()).abs().max())
        assert err <= gtol * scale + 1e-12, (k, err / max(scale, 1e-300))


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------
def test_attentive_pooler_fp32_backward_wiring_matches_reference_autograd(monkeypatch):
    """_AttentivePoolFn in fp32 compute (no autocast): grad mode no longer raises, and with the kernels emulated the gradients of all 19
    parameters match torch autograd through the reference AttentivePooler."""
    import merv_b200 as M

    kernel_emulation.emulate(monkeypatch)
    r = _perturbed_reference(64, 48, 8, 2, 3, "gelu-mlp", 11)
    m = M.AttentivePooler.from_reference(copy.deepcopy(r))
    g = torch.Generator().manual_seed(5)
    x = torch.randn((2, 3, 9, 64), generator=g)
    G = torch.randn((2, 3 * 8, 48), generator=g)
    out = m(x)
    assert out.dtype == torch.float32 and out.requires_grad
    out.backward(G)
    want = r(x)
    want.backward(G)
    assert O.rel_err(out.detach().double().numpy(), want.detach().double().numpy()) < 1e-5
    assert _grads_within(m, r, 1e-4) == 19


def _abi_call(lib, dtype, hd=40, n_q=65, n_kv=70, heads=2, batches=3, ptr=256, ld_short=0, ld_off=0, ws=True, ws_floats=None,
              null=None):
    """merv_cross_attention_backward_ex with fake, never dereferenced pointers: every case below fails before a device is touched."""
    C_ = heads * hd
    need = lib.merv_cross_attention_backward_ex_workspace(batches, n_q, n_kv, heads, hd, dtype)
    p = [ptr] * 5
    if null is not None:
        p[null] = None
    return lib.merv_cross_attention_backward_ex(p[0], C_ + ld_off, 0, p[1], 2 * C_ - ld_short, p[2], C_, p[3], C_, p[4], 2 * C_, batches, n_q,
                                                n_kv, heads, hd, 0.1, dtype, ctypes.c_void_p(4096) if ws else None,
                                                need if ws_floats is None else ws_floats, None)


def test_cross_attention_backward_ex_workspace_and_argument_checks(monkeypatch):
    from merv_b200 import _lib

    lib = _lib.load()
    F32, BF16 = _lib.MERV_F32, _lib.MERV_BF16
    ws = lib.merv_cross_attention_backward_ex_workspace
    monkeypatch.delenv("MERV_ATTN_IMPL", raising=False)
    assert ws(3, 64, 256, 8, 128, BF16) == 0  # the tcgen05 tile needs none
    assert ws(3, 65, 256, 8, 128, BF16) == 3 * 8 * 65 * (128 + 3)  # (m, l, D) and the fp32 dQ per (frame, head, query)
    assert ws(3, 64, 257, 8, 128, BF16) == 3 * 8 * 64 * 131
    assert ws(3, 64, 256, 8, 40, BF16) == 3 * 8 * 64 * 43
    assert ws(3, 64, 256, 8, 128, F32) == 3 * 8 * 64 * 131
    assert ws(0, 64, 256, 8, 128, F32) == 0 and ws(3, 0, 256, 8, 128, F32) == 0
    monkeypatch.setenv("MERV_ATTN_IMPL", "simt")
    assert ws(3, 64, 256, 8, 128, BF16) == 3 * 8 * 64 * 131
    monkeypatch.delenv("MERV_ATTN_IMPL")

    for dt in (F32, BF16):
        for i in range(5):
            assert _abi_call(lib, dt, null=i) == -6, i  # NULL operand
        assert _abi_call(lib, dt, hd=0) == -1
        assert _abi_call(lib, dt, hd=129) == -1
        assert _abi_call(lib, dt, hd=136) == -1 and b"head_dim" in lib.merv_last_error()  # > 128
        assert _abi_call(lib, dt, hd=42) == -1  # not a multiple of the 16-byte vector
        assert _abi_call(lib, dt, ld_short=1) == -1 and b"leading" in lib.merv_last_error()
        assert _abi_call(lib, dt, ld_off=2) == -2  # ldq not a whole number of 16-byte vectors
        assert _abi_call(lib, dt, ptr=260) == -2  # misaligned rows
        assert _abi_call(lib, dt, ws_floats=1) == -6 and b"workspace" in lib.merv_last_error()
    assert _abi_call(lib, F32, ws=False) == -6  # fp32 always runs the CUDA-core kernel, which needs its workspace
    assert _abi_call(lib, 7) == -3  # unknown dtype
