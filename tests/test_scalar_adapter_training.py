"""Training the scalar mixer (``feature_fusion="scalar"``, ScalarAdapter, nn_utils.py:524-537): w = softmax(scalar) for every video,
out = sum_e w_e V_e.

GPU (``-m gpu``): ``ops.scalar_mix_backward`` against fp64 autograd through the reference ScalarAdapter, whole ``MervFusion`` training steps
(fused and module by module) against fp64 autograd through the reference modules, fused against module-by-module gradients,
bit-reproducibility, and an optimizer step followed by an inference forward.  CPU: the autograd wiring with the kernels replaced by torch
restatements of their contracts, the defer policy of linked projectors, and the ABI-level argument checks of the new entry points.
Tolerances (max|a-b| / max|b|): fp32 2e-4, bf16 3e-2 against references at the bf16-rounded operating point.
"""
import ctypes

import pytest
import torch

from oracle import cases as C
from oracle import fusion_oracle as O
from oracle.ref_loader import load_reference_nn_utils
from tests import kernel_emulation

DEV = "cuda:0"
TOL = {torch.float32: 2e-4, torch.bfloat16: 3e-2}
OFFSETS = (0.0, 0.5, -0.5, 0.25)


def _np(t):
    return t.detach().double().cpu().numpy()


def _round(t, dtype):
    return t if dtype == torch.float32 else t.to(torch.bfloat16).float()


def _err(a, b):
    return O.rel_err(_np(a), _np(b))


# ---- the kernel -----------------------------------------------------------------------------------------------------------------------
# (B, T, K): the scalar_mixer golden case (2 videos, 4 x 4 x 4 = 64 tokens, llm_dim 128), K that is not a multiple of a CTA's 128-byte
# column block in either dtype, T that is not a multiple of the 32 token groups, a merv-full-sized case, and a rank without videos
KERNEL_CASES = {"golden": (2, 64, 128), "ragged_k": (3, 48, 200), "ragged_t": (2, 37, 256), "merv_full": (2, 1024, 4096), "no_videos": (0, 64, 128)}


def _kernel_case(name, dtype):
    B, T, K = KERNEL_CASES[name]
    case = C.CASES["scalar_mixer"]
    assert name != "golden" or (B, T, K) == (case.batch, case.token_length, case.llm_dim)
    scalar = torch.from_numpy(C.make_fusion_params(case)["scalar"])
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    V = [_round(torch.randn(B, T, K, generator=g) + OFFSETS[e], dtype) for e in range(4)]
    G = _round(torch.randn(B, T, K, generator=g), dtype)
    H = torch.randn(1, 4, generator=g)
    return scalar, V, G, H


def _reference_kernel_grads(scalar, V, G, H):
    """fp64 autograd of the reference ScalarAdapter for loss = sum(out * G) + sum(w * H): (dV list, dscalar)."""
    ref = load_reference_nn_utils().ScalarAdapter(4).to(device=DEV, dtype=torch.float64)
    with torch.no_grad():
        ref.scalar.copy_(scalar.double())
    leaves = [v.to(DEV).double().requires_grad_(True) for v in V]
    out, w = ref(leaves)
    ((out * G.to(DEV).double()).sum() + (w * H.to(DEV).double()).sum()).backward()
    return [x.grad for x in leaves], ref.scalar.grad


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("name", list(KERNEL_CASES))
def test_scalar_mix_backward_matches_reference_autograd(name, dtype):
    from merv_b200 import ops

    scalar, V, G, H = _kernel_case(name, dtype)
    want_dV, want_ds = _reference_kernel_grads(scalar, V, G, H)
    w, _ = ops.softmax_weights(scalar.to(DEV).reshape(1, 4))
    Vs = [v.to(DEV).to(dtype) for v in V]
    dVs, dscalar = ops.scalar_mix_backward(Vs, G.to(DEV).to(dtype), w.reshape(-1), H.to(DEV).reshape(-1))
    assert dscalar.dtype == torch.float32 and dscalar.shape == (4,)
    assert _err(dscalar, want_ds) < TOL[dtype]
    for e, (g, r) in enumerate(zip(dVs, want_dV)):
        assert g.shape == Vs[e].shape and g.dtype == dtype
        if g.numel():
            assert _err(g, r) < TOL[dtype], f"dV_{e}"


# ---- whole training steps ---------------------------------------------------------------------------------------------------------------
# four encoders (the reference always holds four scalars), 4 frames of 8 x 8 patches pooled to 4 x 4 x 4 = 64 tokens (T % 64 == 0, so the
# fused step applies), llm_dim 128
_DIMS, _TEMPORAL, _H, _LLM, _PTL, _B = [64, 48, 32, 40], [4, 4, 4, 4], 8, 128, 16, 2
STEP_CONFIGS = {  # name: (arch_specifier, fused_training, expected autograd Function of the mix)
    "3davg_linear_fused": ("3davg+linear", True, "_FusedScalarLinearFn"),
    "3davg_linear_module": ("3davg+linear", False, "_ScalarMixFn"),
    "3davg_linear_default": ("3davg+linear", None, None),  # automatic: fused in bf16, module by module in fp32
    "3davg_gelu": ("3davg+gelu-mlp", None, "_ScalarMixFn"),
    "avg_linear": ("avg+linear", None, None),  # fused in bf16, module by module in fp32 (the fused step is bf16 only)
    "3dconv_linear": ("3dconv+linear", None, "_ScalarMixFn"),
}


def _reference_modules(arch):
    """The reference projectors and ScalarAdapter, constructed in MERV.__init__'s order (merv.py:87-227) from the same seed."""
    import functools

    ref = load_reference_nn_utils()
    torch.manual_seed(_DIMS[0])  # merv.py:87
    mlp_type = "linear" if arch.endswith("linear") else "gelu-mlp"
    parts = arch.split("+")
    P = (functools.partial(ref.Convolutional3DProjector, output_size=4) if "3dconv" in parts else
         functools.partial(ref.AveragePooling3DProjector, output_size=4) if "3davg" in parts else functools.partial(ref.AveragePoolingProjector, output_size=4))
    projs = [P(c, _LLM, output_frames=t, mlp_type=mlp_type) for c, t in zip(_DIMS, _TEMPORAL)]
    return projs, ref.ScalarAdapter(len(_DIMS))


def _step_setup(cfg, dtype, device, fused_training="config"):
    """(MervFusion, reference projectors, reference mixer, features, G, H) on one set of bf16-rounded (if needed) parameters and inputs."""
    import merv_b200 as M

    arch, ft, _ = STEP_CONFIGS[cfg]
    ft = ft if fused_training == "config" else fused_training
    m = M.MervFusion.from_config(_DIMS, _LLM, _TEMPORAL, arch_specifier=arch, feature_fusion="scalar", projector_token_length=_PTL,
                                 visual_feature_length=_TEMPORAL[0] * _PTL, fused_training=ft)
    projs, ff = _reference_modules(arch)
    with torch.no_grad():
        m.feature_fusion.scalar.copy_(torch.tensor([0.7, -0.4, 0.1, 0.3]))
        for p in m.parameters():
            p.copy_(_round(p, dtype))
    for p, r in zip(m.projectors, projs):
        r.load_state_dict(p.state_dict())
    ff.load_state_dict(m.feature_fusion.state_dict())
    m = m.to(device=device, dtype=dtype).train()
    g = torch.Generator().manual_seed(3)
    xs = [_round(torch.randn(_B, t, _H * _H, c, generator=g) + 0.2 * i, dtype) for i, (c, t) in enumerate(zip(_DIMS, _TEMPORAL))]
    G = _round(torch.randn(_B, _TEMPORAL[0] * _PTL, _LLM, generator=g), dtype)
    H = torch.randn(1, len(_DIMS), generator=g)
    return m, projs, ff, xs, G, H


def _train_step(m, xs, G, H, device, dtype):
    """One forward + backward of loss = sum(out * G) + sum(w * H); returns (out, w, {name: grad})."""
    m.zero_grad(set_to_none=True)
    out, w = m([x.to(device=device, dtype=dtype) for x in xs])
    ((out.float() * G.to(device)).sum() + (w.float() * H.to(device)).sum()).backward()
    return out, w, {k: p.grad for k, p in m.named_parameters()}


def _check_step(cfg, dtype, device):
    m, projs, ff, xs, G, H = _step_setup(cfg, dtype, device)
    # reference: fp64 autograd through the reference modules, glued as ScalarAdapter's own forward
    projs = [p.double() for p in projs]
    ff = ff.double()
    want_out, want_w = ff([p(x.double()) for p, x in zip(projs, xs)])
    ((want_out * G.double()).sum() + (want_w * H.double()).sum()).backward()

    out, w, grads = _train_step(m, xs, G, H, device, dtype)
    expected = STEP_CONFIGS[cfg][2] or ("_FusedScalarLinearFn" if dtype == torch.bfloat16 else "_ScalarMixFn")
    assert type(out.grad_fn).__name__.startswith(expected)
    tol = TOL[dtype]
    assert w.shape == (1, 4) and _err(out, want_out) < tol and _err(w, want_w) < tol
    want = {f"projectors.{i}.{k}": p.grad for i, r in enumerate(projs) for k, p in r.named_parameters()}
    want["feature_fusion.scalar"] = ff.scalar.grad
    assert sorted(grads) == sorted(want)
    for k, r in want.items():
        assert grads[k] is not None and grads[k].dtype == dtype and _err(grads[k], r) < tol, k
    return grads


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("cfg", list(STEP_CONFIGS))
def test_training_step_matches_reference_autograd(cfg, dtype):
    if cfg == "3davg_linear_fused" and dtype == torch.float32:
        pytest.skip("the fused step is bf16 only; fp32 trains module by module (3davg_linear_module)")
    _check_step(cfg, dtype, DEV)


@pytest.mark.gpu
def test_fused_and_module_by_module_gradients_agree():
    grads = {}
    for ft in (True, False):
        m, _, _, xs, G, H = _step_setup("3davg_linear_fused", torch.bfloat16, DEV, fused_training=ft)
        out, _, grads[ft] = _train_step(m, xs, G, H, DEV, torch.bfloat16)
        assert type(out.grad_fn).__name__.startswith("_FusedScalarLinearFn" if ft else "_ScalarMixFn")
    for k in grads[True]:
        assert _err(grads[True][k], grads[False][k]) < 3e-2, k


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False], ids=["fused", "module"])
def test_training_step_is_bit_reproducible(fused):
    m, _, _, xs, G, H = _step_setup("3davg_linear_fused", torch.bfloat16, DEV, fused_training=fused)
    first = {k: g.clone() for k, g in _train_step(m, xs, G, H, DEV, torch.bfloat16)[2].items()}
    second = _train_step(m, xs, G, H, DEV, torch.bfloat16)[2]
    for k in first:
        assert torch.equal(first[k], second[k]), k


@pytest.mark.gpu
def test_optimizer_step_reaches_the_next_inference_forward():
    """An SGD step after a fused training step: the fused inference forward reads the new scalar and the new projector weights."""
    import merv_b200 as M

    m, _, _, xs, G, H = _step_setup("3davg_linear_fused", torch.bfloat16, DEV)
    xs = [x.to(DEV).to(torch.bfloat16) for x in xs]
    with torch.no_grad():
        out0, w0 = m(xs)
    _train_step(m, xs, G, H, DEV, torch.bfloat16)
    scalar = m.feature_fusion.scalar
    torch.optim.SGD([{"params": [scalar], "lr": 0.5}, {"params": [p for p in m.parameters() if p is not scalar], "lr": 1e-3}]).step()
    with torch.no_grad():
        out1, w1 = m(xs)
    want_w = torch.softmax(m.feature_fusion.scalar.detach().float(), 0)
    assert not torch.equal(w0, w1) and (w1.float()[0] - want_w).abs().max() < 1e-2
    fresh = M.MervFusion.from_config(_DIMS, _LLM, _TEMPORAL, arch_specifier="3davg+linear", feature_fusion="scalar", projector_token_length=_PTL,
                                     visual_feature_length=_TEMPORAL[0] * _PTL)
    fresh.load_state_dict(m.state_dict())
    fresh = fresh.to(device=DEV, dtype=torch.bfloat16).eval()
    with torch.no_grad():
        out2, w2 = fresh(xs)
    assert not torch.equal(out0, out1) and torch.equal(out1, out2) and torch.equal(w1, w2)


# ---- CPU: the autograd wiring with the kernels emulated ----------------------------------------------------------------------------------
def _scalar_mix_backward_standin(Vs, dout, weights, dweights=None):
    """merv_scalar_mix_backward's contract (include/merv_fusion.h) restated with torch ops."""
    dt = Vs[0].dtype
    g = torch.stack([(dout.float() * v.float()).sum() for v in Vs])
    if dweights is not None:
        g = g + dweights
    return [(w * dout.float()).to(dt) for w in weights], weights * (g - (weights * g).sum())


def _scalar_fused_backward_standin(weights, dweights, gsum, dw_partials, biases):
    """merv_scalar_fused_backward's contract (include/merv_fusion.h) restated with torch ops."""
    gs = gsum.sum(0)
    g = torch.stack([p.sum() + (b.float() @ gs if b is not None else 0.0) for p, b in zip(dw_partials, biases)])
    if dweights is not None:
        g = g + dweights
    return weights * (g - (weights * g).sum()), [None if b is None else (w * gs).to(b.dtype) for w, b in zip(weights, biases)]


@pytest.mark.parametrize("cfg,dtype", [("3davg_linear_fused", torch.bfloat16), ("3davg_linear_module", torch.float32),
                                       ("3davg_linear_default", torch.bfloat16), ("3davg_gelu", torch.float32),
                                       ("avg_linear", torch.float32), ("avg_linear", torch.bfloat16)])
def test_training_wiring_matches_reference_on_cpu(cfg, dtype, monkeypatch):
    """The module code unchanged, the kernels emulated: the expected Function is reached and the gradients are the reference's."""
    from merv_b200 import ops

    kernel_emulation.emulate(monkeypatch)
    calls = []

    def spy(name, fn):
        def wrapped(*a, **kw):
            calls.append(name)
            return fn(*a, **kw)
        return wrapped

    monkeypatch.setattr(ops, "scalar_mix_backward", spy("mix", _scalar_mix_backward_standin))
    monkeypatch.setattr(ops, "scalar_fused_backward", spy("fused", _scalar_fused_backward_standin))
    _check_step(cfg, dtype, "cpu")
    fused = STEP_CONFIGS[cfg][2] == "_FusedScalarLinearFn" or (STEP_CONFIGS[cfg][2] is None and dtype == torch.bfloat16)
    assert calls == ["fused" if fused else "mix"]


def test_unequal_encoder_shapes_are_rejected_in_training(monkeypatch):
    """The reference stacks the encoders, so a single-token encoder cannot be trained; inference still broadcasts it."""
    import merv_b200 as M

    kernel_emulation.emulate(monkeypatch)
    ff = M.ScalarAdapter()
    V = [torch.randn(2, 8, 16) for _ in range(3)] + [torch.randn(2, 1, 16)]
    with torch.no_grad():
        out, w = ff(V)
    assert out.shape == (2, 8, 16) and w.shape == (1, 4)
    with pytest.raises(ValueError, match="one \\[B, T, K\\] shape"):
        ff(V)


def test_no_videos_still_trains_the_scalar_on_cpu(monkeypatch):
    import merv_b200 as M
    from merv_b200 import ops

    kernel_emulation.emulate(monkeypatch)
    monkeypatch.setattr(ops, "scalar_mix_backward", _scalar_mix_backward_standin)
    ff = M.ScalarAdapter()
    out, w = ff([torch.empty(0, 8, 16) for _ in range(4)])
    assert out.shape == (0, 8, 16) and w.shape == (1, 4)
    H = torch.randn(1, 4)
    (w * H).sum().backward()
    p = torch.softmax(ff.scalar.detach(), 0)
    assert torch.allclose(ff.scalar.grad, p * (H[0] - (p * H[0]).sum()), atol=1e-6)


# ---- CPU: the defer policy ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("grad", [True, False], ids=["grad", "no_grad"])
def test_fsdp_managed_projector_does_not_defer_to_the_scalar_mixer(grad, monkeypatch):
    import merv_b200 as M

    kernel_emulation.emulate(monkeypatch)
    m = M.MervFusion.from_config(_DIMS, _LLM, _TEMPORAL, arch_specifier="3davg+linear", feature_fusion="scalar", projector_token_length=_PTL,
                                 visual_feature_length=_TEMPORAL[0] * _PTL)
    x = torch.randn(1, _TEMPORAL[0], _H * _H, _DIMS[0])
    p0, ff = m.projectors[0], m.feature_fusion
    with torch.set_grad_enabled(grad):
        assert ff._may_defer(p0) and isinstance(p0(x), M.DeferredProjection)
        p0.projector.projector.weight._fsdp_flattened = True  # what FSDP1 marks a managed parameter with
        assert not ff._may_defer(p0) and isinstance(p0(x), torch.Tensor)
        assert ff._may_defer(m.projectors[1])  # only the managed projector's own unit is affected
        ff.fused_training = True  # projectors and mixer share one FSDP unit
        assert ff._may_defer(p0) and isinstance(p0(x), M.DeferredProjection)
        ff.fused_training = False
        assert not ff._may_defer(p0)


def test_fused_training_is_accepted_for_the_scalar_mixer():
    import merv_b200 as M

    for ft in (True, False):
        m = M.MervFusion.from_config(_DIMS, _LLM, _TEMPORAL, arch_specifier="3davg+linear", feature_fusion="scalar", projector_token_length=_PTL,
                                     visual_feature_length=_TEMPORAL[0] * _PTL, fused_training=ft)
        assert isinstance(m.feature_fusion, M.ScalarAdapter) and m.feature_fusion.fused_training is ft
        m2 = M.MervFusion(list(m.projectors), M.ScalarAdapter(), fused_training=ft)
        assert m2.feature_fusion.fused_training is ft
    assert M.ScalarAdapter().fused_training is None


# ---- CPU: argument checks of the new entry points ----------------------------------------------------------------------------------------
def test_scalar_mix_backward_argument_checks():
    """Checks that run before any device is touched: each returns its MERV_E_* code and names the problem."""
    from merv_b200 import _lib

    lib = _lib.load()
    B, E, T, K = 2, 4, 16, 64
    n = lib.merv_scalar_mix_backward_workspace(B, E, K)
    assert n == B * E * ((K + 31) // 32) and lib.merv_scalar_mix_backward_workspace(0, E, K) == 0
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below fails its checks first
    ptrs = _lib.ptr_array([256] * 9)

    def call(V=ptrs, dOut=fake, weights=fake, dV=ptrs, dscalar=fake, ws=fake, ws_n=n, E=E, K=K, dtype=_lib.MERV_BF16):
        return lib.merv_scalar_mix_backward(V, dOut, weights, None, dV, dscalar, ws, ws_n, B, E, T, K, dtype, None)

    assert call(weights=None) == -6 and b"NULL" in lib.merv_last_error()
    assert call(dscalar=None) == -6
    assert call(V=_lib.ptr_array([256, 0, 256, 256])) == -6 and b"encoder 1" in lib.merv_last_error()
    assert call(dOut=ctypes.c_void_p(264)) == -2 and b"aligned" in lib.merv_last_error()
    assert call(dV=_lib.ptr_array([256, 256, 264, 256])) == -2 and b"encoder 2" in lib.merv_last_error()
    assert call(K=60) == -1 and b"multiple of 8" in lib.merv_last_error()
    assert call(E=9) == -6 and b"E=9" in lib.merv_last_error()
    assert call(ws_n=n - 1) == -6 and b"workspace too small" in lib.merv_last_error()
    assert call(dtype=7) == -3


def test_scalar_fused_backward_argument_checks():
    from merv_b200 import _lib

    lib = _lib.load()
    E, K, B = 4, 128, 2
    n = lib.merv_scalar_fused_backward_workspace(E, K)
    assert n == E * ((K + 255) // 256)
    fake = ctypes.c_void_p(256)
    ptrs = _lib.ptr_array([256] * 9)

    def call(weights=fake, gsum=fake, parts=ptrs, dscalar=fake, ws=fake, ws_n=n, E=E, dtype=_lib.MERV_BF16):
        return lib.merv_scalar_fused_backward(weights, None, gsum, parts, ptrs, ptrs, dscalar, ws, ws_n, B, E, K, dtype, None)

    assert call(weights=None) == -6 and b"NULL" in lib.merv_last_error()
    assert call(gsum=None) == -6 and b"gsum" in lib.merv_last_error()
    assert call(parts=_lib.ptr_array([256, 256, 256, 0])) == -6 and b"encoder 3" in lib.merv_last_error()
    assert call(E=9) == -6 and b"E=9" in lib.merv_last_error()
    assert call(ws_n=n - 1) == -6 and b"workspace too small" in lib.merv_last_error()
    assert call(dtype=7) == -3
