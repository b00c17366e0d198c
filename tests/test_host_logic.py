"""Host-side logic of ``merv_b200/nn_utils.py`` on CPU (``pytest -m "not gpu"``).

The product has no CPU path.  These tests swap the entry points of ``merv_b200.ops`` for the torch stand-ins of
``tests/kernel_emulation.py`` (the CONTRACT of each C entry point, restated) and then run the unmodified module code: which
entry point is called with which tensors, the caches, the deferred/fused plumbing, the autograd wiring of the hand-written
backward, ``patch_merv``.  Outputs are compared with the goldens recorded from the reference, so a wiring mistake shows up
here before it costs GPU time; the kernels themselves are only ever checked on the GPU (tests/test_gpu_parity.py).
"""
import os

import numpy as np
import pytest
import torch

from oracle import cases as C
from oracle import fusion_oracle as O
from tests import kernel_emulation
from tests.golden_util import regenerate
from tests.variant_util import build_variant_module, run_variant

FP32_TOL = 1e-5


@pytest.fixture(autouse=True)
def _emulated(monkeypatch):
    kernel_emulation.emulate(monkeypatch)


def _np(t):
    return t.detach().float().numpy()


def _build(case, pp, fp, dtype, fused):
    import merv_b200 as M

    if case.resampler == "avg":
        projs = [M.AveragePoolingProjector(c, case.llm_dim, case.out_size, t, case.mlp_type) for c, t in zip(case.dims, case.out_frames)]
    else:
        projs = [M.AveragePooling3DProjector(c, case.llm_dim, t, case.out_size, case.mlp_type) for c, t in zip(case.dims, case.out_frames)]
    if case.fusion == "scalar":
        fusion = M.ScalarAdapter(case.num_encoders)
    elif case.fusion == "concat_channel":
        fusion = M.ConcatChannelFusion(case.num_encoders, case.llm_dim)
    else:
        fusion = M.CrossAttentionAdapterLearnableQuery(case.embed_dim, case.llm_dim, case.token_length, averagetoken=True, num_encoder=case.num_encoders)
    m = M.MervFusion(projs, fusion, fused=fused)
    for proj, p in zip(m.projectors, pp):
        proj.projector.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    m.feature_fusion.load_state_dict({k: torch.from_numpy(v) for k, v in fp.items()})
    return m.to(dtype).eval().requires_grad_(False)


SMALL = ["tiny_linear", "tiny_gelu", "tiny_fused_gelu", "frame_factor2", "ragged_windows", "single_encoder", "avg2d_linear", "scalar_mixer",
         "concat_channel"]


@pytest.mark.parametrize("name", SMALL)
def test_module_by_module_wiring_fp32(name):
    case = C.CASES[name]
    g, feats, pp, fp = regenerate(case)
    m = _build(case, pp, fp, torch.float32, fused=False)
    with torch.inference_mode():
        out, w = m([torch.from_numpy(f) for f in feats])
    assert out.shape == (case.batch, case.token_length, case.llm_dim)
    idx = g["sample_idx"]
    assert np.abs(_np(out).reshape(-1)[idx] - g["out_samples"]).max() / float(g["out_abs_max"]) < 2e-5
    if w is not None:
        assert np.abs(_np(w) - g["weights"]).max() < 2e-5


@pytest.mark.parametrize("name", ["tiny_linear", "tiny_gelu", "frame_factor2", "scalar_mixer"])
def test_fused_wiring_bf16(name):
    # the linked path (DeferredProjection -> scores from the last layer's input -> one segmented GEMM) needs bf16 tensors
    case = C.CASES[name]
    if any(c % 8 for c in case.dims):
        pytest.skip("bf16 path needs C % 8 == 0")
    g, feats, pp, fp = regenerate(case)
    m = _build(case, pp, fp, torch.bfloat16, fused=True)
    with torch.inference_mode():
        out, w = m([torch.from_numpy(f).to(torch.bfloat16) for f in feats])
    idx = g["sample_idx"]
    assert np.abs(_np(out).reshape(-1)[idx] - g["out_samples"]).max() / float(g["out_abs_max"]) < 2e-2
    assert np.abs(_np(w) - g["weights"]).max() < 2e-2


# ---- configuration variants -----------------------------------------------------------------------------------
def _variants():
    from oracle import variants as V

    return [n for n in V.VARIANTS if not n.endswith("_wide") and n != "attntv_hd96"]  # the big ones run on the GPU only


@pytest.mark.parametrize("name", _variants())
def test_variant_wiring_fp32(name):
    mod, v, inputs, gold = build_variant_module(name)
    with torch.inference_mode():
        out, w = run_variant(mod, v, inputs)
    assert tuple(out.shape) == gold["out"].shape
    assert O.rel_err(_np(out), gold["out"]) < 2e-5
    if w is not None:
        assert np.abs(_np(w) - gold["weights"]).max() < 2e-5


def test_concat_channel_ln_accepts_the_concatenated_tensor():
    mod, v, inputs, gold = build_variant_module("concat_channel_ln")
    with torch.inference_mode():
        out, _ = run_variant(mod, v, inputs, as_list=False)  # what the unmodified glue passes (merv.py:603-606)
    assert O.rel_err(_np(out), gold["out"]) < 2e-5
    assert sorted(mod.state_dict()) == ["0.bias", "0.weight", "1.projector.bias", "1.projector.weight"]


def test_positional_embedding_through_the_linked_path():
    # pe folds into the per-encoder score constants of the fused path: linked and module-by-module must agree
    import merv_b200 as M

    torch.manual_seed(3)
    dims, K, T, S = [16, 24, 16], 32, 2, 2
    outs = []
    for fused in (False, True):
        torch.manual_seed(5)
        projs = [M.AveragePooling3DProjector(c, K, T, S, "linear") for c in dims]
        ff = M.CrossAttentionAdapterLearnableQuery(24, K, T * S * S, averagetoken=True, num_encoder=3, positional_embedding=True)
        with torch.no_grad():
            ff.Q.mul_(20.0)
            ff.pe.mul_(6.0)
        m = M.MervFusion(projs, ff, fused=fused).to(torch.bfloat16).eval().requires_grad_(False)
        g = torch.Generator().manual_seed(11)
        xs = [torch.randn(2, 4, 16, c, generator=g).to(torch.bfloat16) for c in dims]
        with torch.inference_mode():
            outs.append(m(xs))
    (o0, w0), (o1, w1) = outs
    assert (w0.float() - w1.float()).abs().max() < 2e-2 and (o0.float() - o1.float()).abs().max() < 2e-2 * o0.float().abs().max()
    assert (w0.float() - 1 / 3).abs().max() > 0.02  # the softmax is not flat, so the constants matter


@pytest.mark.parametrize("name", ["pre_ln_linear", "pre_ln_gelu", "pre_ln_deep", "pre_ln_fused_gelu"])
def test_pre_layernorm_backward_wiring(name):
    # _ProjectorFn with the LayerNorm in front: parameter gradients vs torch autograd through the reference's op sequence
    mod, v, inputs, _ = build_variant_module(name)
    mod.requires_grad_(True).train()
    x = torch.from_numpy(inputs[0])
    y = mod(x)
    g = torch.Generator().manual_seed(1)
    dy = torch.randn(y.shape, generator=g)
    y.backward(dy)
    got = {k: p.grad.clone() for k, p in mod.named_parameters()}
    assert all(gr is not None for gr in got.values())
    # same parameters through plain torch modules
    ref_ln = torch.nn.LayerNorm(v["vision_dim"])
    ref_ln.load_state_dict(mod.layernorm.state_dict())
    seq = mod.projector
    params = list(ref_ln.parameters()) + list(seq.parameters())
    for p in params:
        p.grad = None
    seq(ref_ln(x)).backward(dy)
    want = {**{"layernorm." + k: p.grad for k, p in ref_ln.named_parameters()}, **{"projector." + k: p.grad for k, p in seq.named_parameters()}}
    for k in got:
        scale = float(want[k].abs().max()) + 1e-12
        assert float((got[k] - want[k]).abs().max()) / scale < 1e-4, k


def test_projector_input_gradient_when_requested():
    # projected tokens entering concat_channel(_ln) need dX; patch features never do
    import merv_b200 as M

    torch.manual_seed(0)
    p = M.LinearProjector(16, 8).train()
    x = torch.randn(3, 5, 16, requires_grad=True)
    dy = torch.randn(3, 5, 8)
    p(x).backward(dy)
    want = dy @ p.projector.weight.detach()
    assert (x.grad - want).abs().max() < 1e-5


def test_first_and_token_concat_fusions():
    import merv_b200 as M

    case = C.CASES["tiny_linear"]
    g, feats, pp, fp = regenerate(case)
    projs = [M.AveragePooling3DProjector(c, case.llm_dim, t, case.out_size, case.mlp_type) for c, t in zip(case.dims, case.out_frames)]
    for proj, p in zip(projs, pp):
        proj.projector.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    xs = [torch.from_numpy(f) for f in feats]
    want = [O.avgpool3d_projector_forward(f, p, t, case.out_size, case.mlp_type) for f, p, t in zip(feats, pp, case.out_frames)]
    first = M.MervFusion(projs, None, fusion_type="first").eval().requires_grad_(False)
    with torch.inference_mode():
        out, w = first(xs)
    assert w is None and O.rel_err(_np(out), want[0]) < 2e-5
    cat = M.MervFusion(projs, None, fusion_type="concat").eval().requires_grad_(False)
    with torch.inference_mode():
        out, w = cat(xs)
    assert w is None and out.shape[1] == sum(y.shape[1] for y in want)
    assert O.rel_err(_np(out), O.token_concat_forward(want)) < 2e-5
    with pytest.raises(AssertionError):
        M.MervFusion(projs, None)


# ---- patch_merv on the reference's own modules ---------------------------------------------------------------------
class _FakeMerv(torch.nn.Module):
    """The attributes of the reference MERV that patch_merv touches (merv.py:152-223)."""

    def __init__(self, projectors, feature_fusion, fusion_type):
        super().__init__()
        self.projectors = torch.nn.ModuleList(projectors)
        self.feature_fusion = feature_fusion
        self.feature_fusion_type = fusion_type


@pytest.mark.parametrize("fusion_type", ["cross_attention_avg_lq", "concat_channel", "concat_channel_ln", "first", "concat"])
def test_patch_merv_shares_parameters_and_reproduces_the_reference(fusion_type):
    import merv_b200 as M
    from oracle.ref_loader import load_reference_nn_utils

    ref = load_reference_nn_utils()
    torch.manual_seed(1024)
    dims, K, T, S, E = [16, 24, 16], 32, 2, 2, 3
    projs = [ref.AveragePooling3DProjector(c, K, T, S, mlp_type="linear") for c in dims]
    if fusion_type == "cross_attention_avg_lq":
        ff = ref.CrossAttentionAdapterLearnableQuery(embed_dim=24, llm_dim=K, token_length=T * S * S, averagetoken=True, num_encoder=E)
    elif fusion_type == "concat_channel":
        ff = ref.LinearProjector(E * K, K)
    elif fusion_type == "concat_channel_ln":
        ff = torch.nn.Sequential(torch.nn.LayerNorm(E * K), ref.LinearProjector(E * K, K))
    else:
        ff = None
    vid = _FakeMerv(projs, ff, fusion_type).eval().requires_grad_(False)
    keys = sorted(vid.state_dict())
    g = torch.Generator().manual_seed(2)
    xs = [torch.randn(2, 4, 16, c, generator=g) for c in dims]

    def glue(v):  # merv.py:587-609
        ys = [p(x) for p, x in zip(v.projectors, xs)]
        if fusion_type == "first":
            return ys[0]
        if fusion_type == "concat":
            return torch.concat(ys, 1)
        if fusion_type.startswith("concat_channel"):
            return v.feature_fusion(torch.concat(ys, -1))
        return v.feature_fusion(ys)[0]

    with torch.no_grad():
        want = glue(vid)
    ptrs = {k: t.data_ptr() for k, t in vid.state_dict().items()}
    M.patch_merv(vid, fused=False)
    assert sorted(vid.state_dict()) == keys
    assert {k: t.data_ptr() for k, t in vid.state_dict().items()} == ptrs, "parameters must be shared, not copied"
    with torch.inference_mode():
        got = glue(vid)
    assert O.rel_err(_np(got), _np(want)) < 2e-5


# ---- fused training step (the fused forward + _FusedLinearFn backward) vs autograd through the reference's op sequence ----
def test_fused_training_gradients_match_reference_autograd():
    from oracle import torch_port

    case = C.CASES["tiny_linear"]
    g, feats, pp, fp = regenerate(case)
    rnd = lambda a: torch.from_numpy(a).to(torch.bfloat16).float().numpy()  # noqa: E731  (the operating point the bf16 modules see)
    feats_r, pp_r, fp_r = [rnd(f) for f in feats], [{k: rnd(v) for k, v in p.items()} for p in pp], {k: rnd(v) for k, v in fp.items()}
    rng = np.random.default_rng(5)
    G = rng.standard_normal((case.batch, case.token_length, case.llm_dim)).astype(np.float32)
    H = rng.standard_normal((case.batch, case.num_encoders)).astype(np.float32)
    tt = lambda d: {k: torch.from_numpy(v).double().requires_grad_(True) for k, v in d.items()}  # noqa: E731
    ppt, fpt = [tt(p) for p in pp_r], tt(fp_r)
    out, w = torch_port.fusion_forward_autograd([torch.from_numpy(f).double() for f in feats_r], ppt, fpt, case.out_frames, case.out_size,
                                                case.mlp_type, case.token_length)
    ((out * torch.from_numpy(G).double()).sum() + (w * torch.from_numpy(H).double()).sum()).backward()

    import merv_b200 as M

    projs = [M.AveragePooling3DProjector(c, case.llm_dim, t, case.out_size, case.mlp_type) for c, t in zip(case.dims, case.out_frames)]
    fusion = M.CrossAttentionAdapterLearnableQuery(case.embed_dim, case.llm_dim, case.token_length, averagetoken=True, num_encoder=case.num_encoders)
    m = M.MervFusion(projs, fusion, fused=True, fused_training=True)
    for proj, p in zip(m.projectors, pp_r):
        proj.projector.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    m.feature_fusion.load_state_dict({k: torch.from_numpy(v) for k, v in fp_r.items()})
    m = m.to(torch.bfloat16).train()
    got_out, got_w = m([torch.from_numpy(f).to(torch.bfloat16) for f in feats_r])
    assert got_out.requires_grad and got_w.requires_grad and type(got_out.grad_fn).__name__.startswith("_FusedLinearFn")
    assert O.rel_err(_np(got_out), out.detach().numpy()) < 2e-2
    ((got_out.float() * torch.from_numpy(G)).sum() + (got_w.float() * torch.from_numpy(H)).sum()).backward()
    tol = 3e-2
    for i, proj in enumerate(m.projectors):
        for k, p in proj.projector.named_parameters():
            assert p.grad is not None and O.rel_err(_np(p.grad), ppt[i][k].grad.numpy()) < tol, (i, k)
    ff = m.feature_fusion
    E = case.embed_dim
    assert O.rel_err(_np(ff.Q.grad), fpt["Q"].grad.numpy()) < tol
    assert O.rel_err(_np(ff.attention.q_proj_weight.grad), fpt["attention.q_proj_weight"].grad.numpy()) < tol
    assert O.rel_err(_np(ff.attention.k_proj_weight.grad), fpt["attention.k_proj_weight"].grad.numpy()) < tol
    assert O.rel_err(_np(ff.attention.in_proj_bias.grad)[:E], fpt["attention.in_proj_bias"].grad.numpy()[:E]) < tol
    assert ff.attention.v_proj_weight.grad is None and ff.attention.out_proj.weight.grad is None


def test_attentive_pooler_init_sequence_and_adoption_match_the_reference():
    # same seed -> same initial parameters (module tree and init order mirror nn_utils.py:182-227); patch_merv adopts the reference module
    import merv_b200 as M
    from oracle.ref_loader import load_reference_nn_utils

    ref = load_reference_nn_utils()
    torch.manual_seed(77)
    r = ref.AttentivePooler(32, 48, num_query_tokens=4, num_heads=4, output_frames=3, mlp_type="gelu-mlp")
    torch.manual_seed(77)
    m = M.AttentivePooler(32, 48, num_query_tokens=4, num_heads=4, output_frames=3, mlp_type="gelu-mlp")
    rs, ms = r.state_dict(), m.state_dict()
    assert list(rs) == list(ms)
    assert all(torch.equal(rs[k], ms[k]) for k in rs)
    x = torch.randn(2, 3, 9, 32)
    with torch.no_grad():
        want = r.eval()(x)
    vid = _FakeMerv([r], None, "first").eval().requires_grad_(False)
    ptrs = {k: t.data_ptr() for k, t in vid.state_dict().items()}
    M.patch_merv(vid)
    assert isinstance(vid.projectors[0], M.AttentivePooler) and {k: t.data_ptr() for k, t in vid.state_dict().items()} == ptrs
    with torch.inference_mode():
        got = vid.projectors[0](x)
    assert O.rel_err(_np(got), _np(want)) < 2e-5
    assert vid.projectors[0].output_token_length == 4 and vid.projectors[0].output_frame_length == 3


def test_fused_training_is_automatic_unless_fsdp_manages_a_parameter():
    import merv_b200 as M

    def grad_fn_name(mark_sharded):
        torch.manual_seed(0)
        m = M.MervFusion.build([16, 24], 32, [2, 2], 4, "linear", text_embedding_dim=24).to(torch.bfloat16).train()
        assert m.feature_fusion.fused_training is None  # automatic
        if mark_sharded:  # what FSDP1 does to the original parameters it flattens
            m.projectors[1].projector.projector.weight._fsdp_flattened = True
        g = torch.Generator().manual_seed(1)
        out, w = m([torch.randn(2, 2, 16, c, generator=g).to(torch.bfloat16) for c in (16, 24)])
        out.float().sum().backward()
        assert all(p.grad is not None for p in m.projectors.parameters())
        return type(out.grad_fn).__name__

    assert grad_fn_name(False).startswith("_FusedLinearFn")
    assert not grad_fn_name(True).startswith("_FusedLinearFn")  # module-by-module autograd path
    # MLP projectors are outside the fused backward: automatic mode falls back to the module-by-module path
    torch.manual_seed(0)
    m = M.MervFusion.build([16, 24], 32, [2, 2], 4, "gelu-mlp", text_embedding_dim=24).to(torch.bfloat16).train()
    g = torch.Generator().manual_seed(1)
    out, w = m([torch.randn(2, 2, 16, c, generator=g).to(torch.bfloat16) for c in (16, 24)])
    assert out.requires_grad and not type(out.grad_fn).__name__.startswith("_FusedLinearFn")


def test_attentive_pooler_backward_wiring_matches_reference_autograd(monkeypatch):
    """Training the `attntv` resampler: _AttentivePoolFn (hand-written backward; every Linear as dW = dY^T X / dX = dY W, the attention
    through cross_attention_backward, the query tokens' gradient summed over the frames) against torch autograd through the UNMODIFIED
    reference AttentivePooler in fp32.  CPU: the kernels are emulated, so this pins the wiring; the kernels are checked on the GPU."""
    import copy

    import merv_b200 as M
    from oracle.ref_loader import load_reference_nn_utils

    kernel_emulation.emulate(monkeypatch)
    ref = load_reference_nn_utils()
    torch.manual_seed(11)
    r = ref.AttentivePooler(64, 48, num_query_tokens=8, num_heads=2, output_frames=3, mlp_type="gelu-mlp")
    with torch.no_grad():  # non-trivial biases / norms / queries (zeros / ones / std 0.02 by default)
        for name, p in r.named_parameters():
            if name.endswith("bias") or "norm" in name:
                p.add_(0.1 * torch.randn_like(p))
        r.query_tokens.mul_(20.0)
    m = M.AttentivePooler.from_reference(copy.deepcopy(r)).to(torch.bfloat16)
    r = r.to(torch.bfloat16).float()  # the same bf16-rounded parameters on both sides
    g = torch.Generator().manual_seed(5)
    x = torch.randn((2, 3, 9, 64), generator=g).to(torch.bfloat16)
    G = torch.randn((2, 3 * 8, 48), generator=g)
    out = m(x)
    assert out.dtype == torch.bfloat16 and out.requires_grad
    out.backward(G.to(torch.bfloat16))
    want = r(x.float())
    want.backward(G)
    assert O.rel_err(_np(out), _np(want)) < 2e-2
    got = dict(m.named_parameters())
    seen = 0
    for name, p in r.named_parameters():
        assert got[name].grad is not None, name
        scale = float(p.grad.abs().max())
        assert float((got[name].grad.float() - p.grad).abs().max()) <= 4e-2 * scale + 1e-6, name
        seen += 1
    assert seen == 19  # query tokens, 2 LayerNorms, kv / q / proj / fc1 / fc2, the 2-layer projector


def test_conv3d_projector_backward_wiring_and_adoption_match_the_reference(monkeypatch):
    """The `3dconv` resampler (Convolutional3DProjector, nn_utils.py:341-377): pooled-taps GEMM forward and its hand-written backward
    (_ConvTapsFn: dW = dY^T A folded back into Conv3d's [K, C, 3, 3, 3], db = colsum) against torch autograd through the UNMODIFIED
    reference module, adopted with from_reference (shared parameters).  CPU: kernels emulated, so this pins the wiring."""
    import copy

    import merv_b200 as M
    from oracle.ref_loader import load_reference_nn_utils

    kernel_emulation.emulate(monkeypatch)
    ref = load_reference_nn_utils()
    torch.manual_seed(3)
    r = ref.Convolutional3DProjector(16, 24, output_frames=2, output_size=3, mlp_type="gelu-mlp")
    m = M.Convolutional3DProjector.from_reference(copy.deepcopy(r))
    assert list(m.state_dict()) == list(r.state_dict())
    assert m.output_token_length == r.output_token_length == 9 and m.output_frame_length == r.output_frame_length == 2
    g = torch.Generator().manual_seed(5)
    x = torch.randn((2, 5, 49, 16), generator=g)
    G = torch.randn((2, 2 * 9, 24), generator=g)
    out = m(x)
    out.backward(G)
    want = r(x)
    want.backward(G)
    assert O.rel_err(_np(out), _np(want)) < 1e-5
    got = dict(m.named_parameters())
    for name, p in r.named_parameters():
        assert got[name].grad is not None and got[name].grad.shape == p.grad.shape, name
        assert float((got[name].grad - p.grad).abs().max()) <= 1e-4 * float(p.grad.abs().max()) + 1e-7, name
    # the tap-major weight view is rebuilt when the parameter changes (version counter), not served stale
    with torch.no_grad():
        y0 = m(x)
        m.convolution_pooling[0].weight.mul_(0.5)
        m.convolution_pooling[0].bias.zero_()
        y1 = m(x)
        r.convolution_pooling[0].weight.mul_(0.5)
        r.convolution_pooling[0].bias.zero_()
        assert O.rel_err(_np(y1), _np(r(x))) < 1e-5 and not torch.equal(y0, y1)
