"""GPU parity tests (B200): every kernel and both module paths, called through the C ABI, against the numpy
oracle on the same seeded inputs and against the golden fixtures recorded from the unmodified reference.

Tolerances (BASELINE.json north_star; metric max|a-b| / max|b|, BASELINE.md §5):
    fp32 : 1e-5      bf16 : 2e-2
"""
import numpy as np
import pytest
import torch

from oracle import cases as C
from oracle import fusion_oracle as O
from tests.golden_util import regenerate

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_TOL = 2e-2
DEV = "cuda:0"


def _t(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV).to(dtype)


def _np(t):
    return t.detach().float().cpu().numpy()


def _bf16_round(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.bfloat16).float().numpy()


def build_module(case, pp, fp, dtype, fused):
    import merv_b200 as M

    if case.resampler == "avg":  # 2-D per-frame resampler (merv.py:116-122)
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
    return m.to(device=DEV, dtype=dtype).eval().requires_grad_(False)


# ---------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["tiny_linear", "frame_factor2", "ragged_windows", "single_encoder", "mid_linear"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("impl", ["tma", "direct"])
def test_pool3d_matches_oracle(name, dtype, impl, monkeypatch):
    from merv_b200 import ops

    if impl == "direct":
        monkeypatch.setenv("MERV_POOL_IMPL", "direct")  # the plain-load fallback kernel
    case = C.CASES[name]
    g, feats, _, _ = regenerate(case)
    vec = 8 if dtype == torch.bfloat16 else 4
    if any(c % vec for c in case.dims):
        pytest.skip("channel count not a multiple of the 16-byte vector for this dtype")
    xs = [_t(f, dtype) for f in feats]
    rng = np.random.default_rng(1)
    svs = [rng.standard_normal(c).astype(np.float32) for c in case.dims]
    ys, partials = ops.pool3d(xs, case.out_frames, case.out_size, score_vecs=[_t(v) for v in svs])
    ys2, none = ops.pool3d(xs, case.out_frames, case.out_size)
    torch.cuda.synchronize()
    assert none is None
    for e, (x, y, pt) in enumerate(zip(xs, ys, partials)):
        want = O.avg_pool3d_tokens(_np(x), case.out_frames[e], case.out_size)  # oracle on the dtype-rounded input
        assert y.shape == want.shape and y.dtype == dtype
        tol = 1e-6 if dtype == torch.float32 else 4e-3  # bf16: one rounding of the fp32 mean
        assert O.rel_err(_np(y), want) < tol
        assert torch.equal(y, ys2[e])
        if name in C.FULL_STORE_CASES and dtype == torch.float32:
            assert O.rel_err(_np(y), g[f"pooled{e}"]) < FP32_TOL
        # deterministic partial dot products of the pooled tokens (as stored) with the score vector
        want_dot = (_np(y).astype(np.float64).sum(1) * svs[e]).sum(-1)
        got = _np(pt).astype(np.float64).sum(1)
        assert pt.shape[0] == case.batch
        assert np.abs(got - want_dot).max() < 2e-4 * max(1.0, np.abs(want_dot).max())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("H,F,T,C", [(16, 4, 4, 192), (14, 4, 4, 192), (16, 8, 4, 64), (14, 6, 4, 200), (14, 5, 3, 72)])
def test_pool3d_square_grid_consumer_matches_oracle(H, F, T, C, dtype):
    # the separable compile-time-window consumer of the TMA kernel (16 x 16 and 14 x 14 patches -> 8 x 8, 128-byte channel slabs):
    # temporal windows of 1, 2 and ragged 1-2 frames, a channel tail that hangs over the last slab, strided frames, score partials
    from merv_b200 import ops

    rng = np.random.default_rng(H * 100 + F * 10 + T)
    B = 3
    full = _t(rng.standard_normal((B, F, H * H + 1, C), dtype=np.float32) + 0.25, dtype)
    x = full[:, :, 1:, :]  # CLS-dropping slice: frame stride (N + 1) * C
    sv = rng.standard_normal(C).astype(np.float32)
    (y,), (pt,) = ops.pool3d([x], [T], 8, score_vecs=[_t(sv)])
    (yd,), _ = ops.pool3d([x.contiguous()], [T], 8)
    torch.cuda.synchronize()
    want = O.avg_pool3d_tokens(_np(x), T, 8)
    assert y.shape == want.shape == (B, T * 64, C) and y.dtype == dtype
    assert O.rel_err(_np(y), want) < (1e-6 if dtype == torch.float32 else 4e-3)
    assert torch.equal(y, yd)
    want_dot = (_np(y).astype(np.float64).sum(1) * sv).sum(-1)
    assert np.abs(_np(pt).astype(np.float64).sum(1) - want_dot).max() < 2e-4 * max(1.0, np.abs(want_dot).max())


def test_pool3d_strided_input_drops_cls_token():
    # backbones hand over slices that drop a CLS token (languagebind/__init__.py:94): token stride stays C,
    # frame stride is (N+1)*C — the kernel must honour strides instead of forcing a copy
    from merv_b200 import ops

    rng = np.random.default_rng(3)
    full = _t(rng.standard_normal((2, 4, 17, 64), dtype=np.float32), torch.bfloat16)
    x = full[:, :, 1:, :]
    assert not x.is_contiguous()
    (y,), _ = ops.pool3d([x], [4], 2)
    want = O.avg_pool3d_tokens(_np(x), 4, 2)
    assert O.rel_err(_np(y), want) < 4e-3


GEMM_SHAPES = [
    (256, 512, 256), (128, 256, 64), (100, 136, 72), (1000, 264, 200), (2048, 4096, 1024), (384, 768, 4096),
]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
@pytest.mark.parametrize("act", [0, 1])
@pytest.mark.parametrize("cta_group", [1, 2])
def test_tcgen05_linear_matches_oracle(M, N, K, act, cta_group, monkeypatch):
    from merv_b200 import ops

    monkeypatch.setenv("MERV_GEMM_CTA_GROUP", str(cta_group))  # single-CTA kernel / CTA-pair (cta_group::2) kernel

    rng = np.random.default_rng(M + N + K)
    a = _bf16_round(rng.standard_normal((M, K), dtype=np.float32))
    w = _bf16_round(rng.uniform(-1, 1, (N, K)).astype(np.float32) / np.sqrt(K))
    b = _bf16_round(rng.uniform(-0.5, 0.5, N).astype(np.float32))
    rv = rng.standard_normal(N).astype(np.float32)
    y, rd = ops.linear_bias_act(_t(a, torch.bfloat16), _t(w, torch.bfloat16), _t(b, torch.bfloat16), act, rowdot_vec=_t(rv))
    torch.cuda.synchronize()
    want = a.astype(np.float64) @ w.astype(np.float64).T + b
    if act:
        want = O.gelu_erf(want)
    assert y.shape == (M, N)
    assert O.rel_err(_np(y), want) < 6e-3  # fp32 accumulate, one bf16 rounding of the output
    # row-dot partials: dot of the STORED row with rv, per MERV_ROWDOT_BLOCK-column block
    from merv_b200._lib import ROWDOT_BLOCK as RB

    nblk = (N + RB - 1) // RB
    yy = _np(y).astype(np.float64)
    want_rd = np.stack([(yy[:, j * RB:(j + 1) * RB] * rv[j * RB:(j + 1) * RB]).sum(1) for j in range(nblk)], 1)
    assert rd.shape == (M, nblk)
    assert np.abs(_np(rd) - want_rd).max() < 1e-3 * max(1.0, np.abs(want_rd).max())


@pytest.mark.parametrize("M,N,K", [(256, 512, 256), (128, 256, 64), (104, 136, 72), (1000, 264, 200), (4096, 1024, 2048), (768, 384, 4997)])
@pytest.mark.parametrize("a_t,w_t", [(True, False), (False, True), (True, True)])
@pytest.mark.parametrize("cta_group", [1, 2])
def test_tcgen05_gemm_with_mn_major_operands_matches_oracle(M, N, K, a_t, w_t, cta_group, monkeypatch):
    """merv_gemm_ex: either operand handed over transposed ([K, M] / [K, N]) and read MN-major by the tensor cores — the forms the
    backward of a Linear needs (dW = dY^T X contracts over the tokens; dX = dY W).  K = 5000 with both operands MN-major: a k tail that
    is not a multiple of 8 (any number of tokens), zero-filled by TMA."""
    from merv_b200 import ops

    if K % 8 and not (a_t and w_t):
        pytest.skip("K % 8 != 0 needs both operands MN-major")
    monkeypatch.setenv("MERV_GEMM_CTA_GROUP", str(cta_group))
    rng = np.random.default_rng(M + 3 * N + 7 * K)
    a = _bf16_round(rng.standard_normal((M, K), dtype=np.float32))
    w = _bf16_round(rng.uniform(-1, 1, (N, K)).astype(np.float32) / np.sqrt(K))
    b = _bf16_round(rng.uniform(-0.5, 0.5, N).astype(np.float32))
    ta = _t(a.T if a_t else a, torch.bfloat16)
    tw = _t(w.T if w_t else w, torch.bfloat16)
    y = ops.gemm_ex(ta, tw, _t(b, torch.bfloat16), 0, a_t=a_t, w_t=w_t)
    torch.cuda.synchronize()
    want = a.astype(np.float64) @ w.astype(np.float64).T + b
    assert y.shape == (M, N)
    assert O.rel_err(_np(y), want) < 6e-3
    # strided views (a column slice of a wider matrix) are read in place
    if a_t and M >= 256:
        wide = _t(np.concatenate([a.T, a.T], 1), torch.bfloat16)  # [K, 2M]
        y2 = ops.gemm_ex(wide[:, M:], tw, _t(b, torch.bfloat16), 0, a_t=True, w_t=w_t)
        assert torch.equal(y2, y)


def test_simt_fp32_linear_matches_oracle():
    from merv_b200 import ops

    rng = np.random.default_rng(5)
    for M, N, K in [(130, 70, 50), (256, 512, 768)]:
        a = rng.standard_normal((M, K), dtype=np.float32)
        w = rng.uniform(-1, 1, (N, K)).astype(np.float32) / np.sqrt(K)
        b = rng.uniform(-0.5, 0.5, N).astype(np.float32)
        for act in (0, 1):
            y, _ = ops.linear_bias_act(_t(a), _t(w), _t(b), act)
            want = a.astype(np.float64) @ w.astype(np.float64).T + b
            if act:
                want = O.gelu_erf(want)
            assert O.rel_err(_np(y), want) < 2e-6


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_query_vector_matches_oracle(dtype):
    from merv_b200 import ops

    case = C.CASES["mid_linear"]
    fp = C.make_fusion_params(case)
    if dtype == torch.bfloat16:
        fp = {k: _bf16_round(v) for k, v in fp.items()}
    u = ops.fusion_query_vec(_t(fp["Q"], dtype), _t(fp["attention.q_proj_weight"], dtype), _t(fp["attention.k_proj_weight"], dtype),
                             _t(fp["attention.in_proj_bias"], dtype))
    want = O.fusion_query_vector({k: v.astype(np.float64) for k, v in fp.items()})
    assert O.rel_err(_np(u), want) < 1e-5


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_mix_kernels_match_oracle_incl_broadcast(dtype):
    # general adapter path on arbitrary tensors, including a T==1 encoder (nn_utils.py:502)
    import merv_b200 as M

    case = C.CASES["mid_linear"]
    fp = C.make_fusion_params(case)
    rng = np.random.default_rng(11)
    T, K, B = case.token_length, case.llm_dim, 3
    V = [rng.standard_normal((B, T, K), dtype=np.float32) + 0.3, rng.standard_normal((B, 1, K), dtype=np.float32),
         rng.standard_normal((B, T, K), dtype=np.float32) - 0.2]
    ff = M.CrossAttentionAdapterLearnableQuery(case.embed_dim, K, T, averagetoken=True, num_encoder=3)
    ff.load_state_dict({k: torch.from_numpy(v) for k, v in fp.items()})
    ff = ff.to(device=DEV, dtype=dtype).eval().requires_grad_(False)
    out, w = ff([_t(v, dtype) for v in V])
    Vr = [_np(_t(v, dtype)) for v in V]
    fpr = {k: _np(_t(v, dtype)) for k, v in fp.items()}
    want_out, want_w = O.cross_attention_fusion_forward([v.astype(np.float64) for v in Vr], {k: v.astype(np.float64) for k, v in fpr.items()}, T)
    tol = FP32_TOL if dtype == torch.float32 else 6e-3
    assert out.shape == (B, T, K) and w.shape == (B, 3) and out.dtype == dtype
    assert np.abs(_np(w) - want_w).max() < (2e-5 if dtype == torch.float32 else 4e-3)
    assert O.rel_err(_np(out), want_out) < tol


# ---------------------------------------------------------------------------------------------------------
# module paths vs the reference goldens
# ---------------------------------------------------------------------------------------------------------
SMALL = ["tiny_linear", "tiny_gelu", "tiny_fused_gelu", "frame_factor2", "ragged_windows", "single_encoder", "mid_linear", "mid_gelu",
         "avg2d_linear", "scalar_mixer", "concat_channel"]


def _check_against_golden(case, g, out, w, tol, wtol):
    assert out.shape == (case.batch, case.token_length, case.llm_dim)
    if case.fusion == "concat_channel":  # no mixing weights (merv.py:603-606: mixer_value stays None)
        assert w is None
        w = torch.zeros((case.batch, 0))
        out_np = _np(out)
        assert np.abs(out_np.reshape(-1)[g["sample_idx"]] - g["out_samples"]).max() / float(g["out_abs_max"]) < tol
        return
    out_np, w_np = _np(out), _np(w)
    assert w.shape == ((1 if case.fusion == "scalar" else case.batch), case.num_encoders)  # ScalarAdapter returns [1, E] (nn_utils.py:537)
    assert np.allclose(w_np.sum(-1), 1.0, atol=1e-2 if wtol > 1e-4 else 1e-5)
    scale = float(g["out_abs_max"])
    idx = g["sample_idx"]
    assert np.abs(out_np.reshape(-1)[idx] - g["out_samples"]).max() / scale < tol
    assert np.abs(w_np - g["weights"]).max() < wtol
    if case.name in C.FULL_STORE_CASES:
        assert O.rel_err(out_np, g["out"]) < tol


@pytest.mark.parametrize("name", SMALL + ["merv_full_b1"])
def test_modules_fp32_match_reference(name):
    case = C.CASES[name]
    if any(c % 4 for c in case.dims):
        pytest.skip("fp32 path needs C % 4 == 0")
    g, feats, pp, fp = regenerate(case)
    m = build_module(case, pp, fp, torch.float32, fused=False)
    with torch.inference_mode():
        out, w = m([_t(f) for f in feats])
    assert out.dtype == torch.float32
    _check_against_golden(case, g, out, w, FP32_TOL, 2e-5)


@pytest.mark.parametrize("name", SMALL + ["merv_full_b1", "merv_full_b1_gelu"])
@pytest.mark.parametrize("fused", [False, True])
def test_modules_bf16_match_reference(name, fused):
    case = C.CASES[name]
    if any(c % 8 for c in case.dims):
        pytest.skip("bf16 path needs C % 8 == 0")
    g, feats, pp, fp = regenerate(case)
    m = build_module(case, pp, fp, torch.bfloat16, fused=fused)
    with torch.inference_mode():
        out, w = m([_t(f, torch.bfloat16) for f in feats])
    assert out.dtype == torch.bfloat16 and out.is_contiguous()
    _check_against_golden(case, g, out, w, BF16_TOL, 2e-2)
    # also against the reference's own bf16 run (what a user switching frameworks would compare with)
    idx = g["sample_idx"]
    assert np.abs(_np(out).reshape(-1)[idx] - g["out_samples_bf16"]).max() / float(g["out_abs_max"]) < BF16_TOL


@pytest.mark.parametrize("name", ["mid_linear", "mid_gelu"])
def test_autocast_fp32_master_weights(name):
    # training-style call: fp32 parameters under torch.autocast(bf16) (base_strategy.py:210-214)
    case = C.CASES[name]
    g, feats, pp, fp = regenerate(case)
    m = build_module(case, pp, fp, torch.float32, fused=True)
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        out, w = m([_t(f, torch.bfloat16) for f in feats])
    assert out.dtype == torch.bfloat16
    _check_against_golden(case, g, out, w, BF16_TOL, 2e-2)


@pytest.mark.parametrize("name", ["mid_linear", "mid_gelu", "merv_full_b1"])
def test_cta_pair_kernel_through_the_modules(name, monkeypatch):
    # the whole fused path with every GEMM forced onto the cta_group::2 kernel
    monkeypatch.setenv("MERV_GEMM_CTA_GROUP", "2")
    case = C.CASES[name]
    g, feats, pp, fp = regenerate(case)
    m = build_module(case, pp, fp, torch.bfloat16, fused=True)
    with torch.inference_mode():
        out, w = m([_t(f, torch.bfloat16) for f in feats])
    _check_against_golden(case, g, out, w, BF16_TOL, 2e-2)


def test_fused_equals_unfused_and_oracle_on_rounded_inputs():
    # isolate kernel error from bf16 input rounding: oracle run in fp64 on the bf16-rounded inputs/weights
    case = C.CASES["mid_linear"]
    g, feats, pp, fp = regenerate(case)
    feats_r = [_bf16_round(f) for f in feats]
    pp_r = [{k: _bf16_round(v) for k, v in p.items()} for p in pp]
    fp_r = {k: _bf16_round(v) for k, v in fp.items()}
    want, want_w, _ = O.merv_fusion_forward([f.astype(np.float64) for f in feats_r], [{k: v.astype(np.float64) for k, v in p.items()} for p in pp_r],
                                            {k: v.astype(np.float64) for k, v in fp_r.items()}, case.out_frames, case.out_size,
                                            case.mlp_type, case.token_length)
    outs = {}
    for fused in (False, True):
        m = build_module(case, pp, fp, torch.bfloat16, fused=fused)
        with torch.inference_mode():
            out, w = m([_t(f, torch.bfloat16) for f in feats])
        outs[fused] = _np(out)
        assert O.rel_err(_np(out), want) < 8e-3
        assert np.abs(_np(w) - want_w).max() < 5e-3
    assert O.rel_err(outs[True], outs[False]) < 8e-3


# ---------------------------------------------------------------------------------------------------------
# size-independent properties at the benchmark shape (merv-full, bf16)
# ---------------------------------------------------------------------------------------------------------
def _full_module(fused=True, mlp_type="linear"):
    import merv_b200 as M

    m = M.MervFusion.build([1024, 1024, 768, 768], 4096, [16] * 4, 64, mlp_type, seed=1024, fused=fused)
    with torch.no_grad():
        m.feature_fusion.Q.mul_(64.0)  # non-degenerate softmax (SURVEY.md §7)
    return m.to(device=DEV, dtype=torch.bfloat16).eval().requires_grad_(False)


def _full_features(B, seed=7):
    g = torch.Generator(device=DEV).manual_seed(seed)
    shapes = [(B, 16, 256, 1024), (B, 16, 256, 1024), (B, 16, 196, 768), (B, 16, 196, 768)]
    mus = [0.0, 0.5, -0.5, 0.25]
    return [(torch.randn(s, generator=g, device=DEV) + mu).to(torch.bfloat16) for s, mu in zip(shapes, mus)]


@pytest.mark.parametrize("fused,B", [(True, 64), (False, 16)])  # B = 64 is BASELINE.json's benchmark batch
def test_full_size_batch_properties(fused, B):
    m = _full_module(fused)
    feats = _full_features(B)
    with torch.inference_mode():
        out, w = m(feats)
        out2, w2 = m(feats)
        torch.cuda.synchronize()
        assert out.shape == (B, 1024, 4096) and w.shape == (B, 4)
        assert torch.isfinite(out.float()).all()
        assert torch.allclose(w.float().sum(-1), torch.ones(B, device=DEV), atol=1e-2)
        assert (w.float().max(-1).values - w.float().min(-1).values).mean() > 0.02, "softmax is degenerate: test would not see a broken score path"
        # determinism: fixed-order reductions, no atomics
        assert torch.equal(out, out2) and torch.equal(w, w2)
        # videos are independent: a video computed alone (as another rank would) is bit-identical
        for b in (0, B - 1):
            ob, wb = m([f[b:b + 1] for f in feats])
            assert torch.equal(ob[0], out[b]) and torch.equal(wb[0], w[b])
        # a contiguous shard equals the same rows of the full batch (what batch-sharding across GPUs relies on)
        oh, wh = m([f[B // 2:] for f in feats])
        assert torch.equal(oh, out[B // 2:]) and torch.equal(wh, w[B // 2:])


def test_benchmark_batch_matches_the_oracle_directly():
    """The exact run bench.py times (merv-full, B = 64, bf16, the single-call production path) checked DIRECTLY against the CPU
    oracle: three videos are pulled out of the batch of 64 and recomputed by oracle.merv_fusion_forward in fp64 from the same
    bf16-rounded inputs and weights (tolerance 2e-2, BASELINE.json) — and, where the staged reference file travelled with the
    snapshot (oracle/_ref), by the unmodified reference modules in fp32."""
    B = 64
    m = _full_module(True)
    feats = _full_features(B)
    with torch.inference_mode():
        out, w = m(feats)      # builds the plan
        out, w = m(feats)      # re-runs the cached single-call plan: what the timed loop of bench.py executes
    torch.cuda.synchronize()
    pp = [{k: _np(v).astype(np.float64) for k, v in p.projector.state_dict().items()} for p in m.projectors]
    fp = {k: _np(v).astype(np.float64) for k, v in m.feature_fusion.state_dict().items()}
    picks = [0, 37, B - 1]
    sub = [_np(f[picks]).astype(np.float64) for f in feats]
    want, want_w, _ = O.merv_fusion_forward(sub, pp, fp, (16, 16, 16, 16), 8, "linear", 1024)
    got, got_w = _np(out[picks]), _np(w[picks])
    assert got.shape == want.shape == (3, 1024, 4096)
    assert O.rel_err(got, want) < BF16_TOL, O.rel_err(got, want)
    assert np.abs(got_w - want_w).max() < 1e-2
    assert (want_w.max(-1) - want_w.min(-1)).mean() > 0.02, "degenerate softmax: the score path would not be exercised"
    from oracle.ref_loader import reference_available

    if reference_available():  # the real reference modules (CPU, fp32) on the same three videos
        from oracle import reference_model

        fwd, (projs, ff) = reference_model.build_reference([1024, 1024, 768, 768], 4096, [16] * 4, 8, "linear", 1024, q_scale=64.0)
        for rp, mp in zip(projs, m.projectors):  # the module under test rounded its seeded fp32 weights to bf16: give the reference those
            rp.projector.load_state_dict({k: v.float().cpu() for k, v in mp.projector.state_dict().items()})
        ff.load_state_dict({k: v.float().cpu() for k, v in m.feature_fusion.state_dict().items()})
        ref_out, ref_w = fwd([f[picks].float().cpu() for f in feats])
        assert O.rel_err(got, ref_out.numpy()) < BF16_TOL
        assert np.abs(got_w - ref_w.numpy()).max() < 1e-2


def test_full_size_fused_matches_unfused():
    B = 4
    feats = _full_features(B, seed=9)
    with torch.inference_mode():
        of, wf = _full_module(True)(feats)
        ou, wu = _full_module(False)(feats)
    scale = ou.float().abs().max().item()
    assert (of.float() - ou.float()).abs().max().item() / scale < 1.2e-2
    assert (wf.float() - wu.float()).abs().max().item() < 1e-2


def test_single_encoder_siglip_config():
    # BASELINE.json config 4: one encoder (SigLIP), E=1 -> weights == 1 and prefix == projected tokens
    import merv_b200 as M

    m = M.MervFusion.build([768], 4096, [16], 64, "linear", seed=768, fused=True).to(device=DEV, dtype=torch.bfloat16).eval().requires_grad_(False)
    mu = M.MervFusion(list(m.projectors), m.feature_fusion, fused=False)
    x = _full_features(2)[3]
    with torch.inference_mode():
        out, w = m([x])
        M.unlink(m.projectors)
        y = m.projectors[0](x)
    assert torch.equal(w.float(), torch.ones_like(w.float()))
    assert (out.float() - y.float()).abs().max().item() / y.float().abs().max().item() < 8e-3
    del mu


# ---------------------------------------------------------------------------------------------------------
# error behaviour mirrors the reference
# ---------------------------------------------------------------------------------------------------------
def test_error_behaviour():
    import merv_b200 as M
    from merv_b200 import _lib, ops

    ff = M.CrossAttentionAdapterLearnableQuery(96, 128, 64, averagetoken=True).to(DEV).eval().requires_grad_(False)
    with pytest.raises(AssertionError):  # nn_utils.py:494-495
        ff([torch.zeros(1, 63, 128, device=DEV)])
    with pytest.raises(TypeError):
        ops.linear_bias_act(torch.zeros(4, 8, device=DEV, dtype=torch.float16), torch.zeros(8, 8, device=DEV, dtype=torch.float16), None)
    with pytest.raises(_lib.MervError, match="MERV_E_ALIGN|MERV_E_SHAPE"):
        ops.linear_bias_act(torch.zeros(4, 12, device=DEV, dtype=torch.bfloat16), torch.zeros(8, 12, device=DEV, dtype=torch.bfloat16), None)
    p = M.AveragePooling3DProjector(64, 128, 4, 4, "linear").to(DEV).requires_grad_(False)
    with pytest.raises(AssertionError):  # 15 patches: not a square grid
        p(torch.zeros(1, 4, 15, 64, device=DEV))


# ---------------------------------------------------------------------------------------------------------
# SURVEY.md §8 f-2 / f-3: prefix written straight into the multimodal embedding buffer; fused batch gather
# ---------------------------------------------------------------------------------------------------------
def test_prefix_written_into_embedding_buffer_and_gather():
    case = C.CASES["mid_linear"]  # T = 128 tokens per video: a multiple of the 128-row GEMM tile
    g, feats, pp, fp = regenerate(case)
    m = build_module(case, pp, fp, torch.bfloat16, fused=True)
    B0, T, K = case.batch, case.token_length, case.llm_dim
    # a batch of 5 "examples" of which rows [3, 0, 3] are multimodal (merv.py:572: patch_feature[multimodal_indices])
    rep = [torch.cat([_t(f, torch.bfloat16)] * 3)[:5].contiguous() for f in feats]  # source batch of 5 videos
    idx = torch.tensor([3, 0, 3], device=DEV)
    text = torch.randn(5, 9, K, device=DEV).to(torch.bfloat16)  # [BOS + 8 text tokens] embeddings
    with torch.inference_mode():
        want_prefix, want_w = m([f[idx] for f in rep])  # gather done by torch, plain output
        buf, w = m.forward_into_embeddings(rep, text, bos_token_length=1, multimodal_indices=idx)
    assert buf.shape == (3, 9 + T, K)
    assert torch.equal(buf[:, 1:1 + T], want_prefix), "prefix written in place must be bit-identical to the plain output"
    assert torch.equal(w, want_w)
    assert torch.equal(buf[:, :1], text[idx][:, :1]) and torch.equal(buf[:, 1 + T:], text[idx][:, 1:])  # merv.py:633-640
    # and against the reference golden (videos 3 and 0 of the repeated batch are golden videos 1 and 0)
    scale = float(g["out_abs_max"])
    idxs = g["sample_idx"]
    got = torch.stack([buf[1, 1:1 + T], buf[0, 1:1 + T]])  # golden order: video 0, video 1  ->  source videos 0, 3
    assert np.abs(_np(got).reshape(-1)[idxs] - g["out_samples"]).max() / scale < BF16_TOL


def test_strided_output_requires_tile_aligned_videos():
    from merv_b200 import _lib, ops

    a = torch.randn(2 * 96, 64, device=DEV).to(torch.bfloat16)
    w = torch.randn(256, 64, device=DEV).to(torch.bfloat16)
    scale = torch.ones(2, 1, device=DEV)
    buf = torch.zeros(2, 100, 256, device=DEV, dtype=torch.bfloat16)
    with pytest.raises(_lib.MervError, match="MERV_E_SHAPE"):  # 96 rows per video is not a multiple of the 128-row tile
        ops.fused_linear_mix([a], [w], scale, None, 96, out=buf[:, 2:98])
    out = ops.fused_linear_mix([a], [w], scale, None, 96)  # contiguous output has no such restriction
    assert O.rel_err(_np(out), _np(a) @ _np(w).T) < 6e-3


# ---------------------------------------------------------------------------------------------------------
# SURVEY.md §8 f-1: backward of the module-by-module path vs torch autograd through the reference's op sequence
# ---------------------------------------------------------------------------------------------------------
def _reference_grads(case, feats, pp, fp, G, H):
    from oracle import torch_port

    tt = lambda d: {k: torch.from_numpy(v).double().requires_grad_(True) for k, v in d.items()}  # noqa: E731
    ppt, fpt = [tt(p) for p in pp], tt(fp)
    out, w = torch_port.fusion_forward_autograd([torch.from_numpy(f).double() for f in feats], ppt, fpt, case.out_frames, case.out_size,
                                                case.mlp_type, case.token_length)
    loss = (out * torch.from_numpy(G).double()).sum() + (w * torch.from_numpy(H).double()).sum()
    loss.backward()
    return [{k: v.grad.numpy() for k, v in p.items()} for p in ppt], {k: (None if v.grad is None else v.grad.numpy()) for k, v in fpt.items()}


@pytest.mark.parametrize("dtype,tol,fused_training", [(torch.float32, 2e-4, False), (torch.bfloat16, 3e-2, False), (torch.bfloat16, 3e-2, True)])
@pytest.mark.parametrize("name", ["mid_linear", "mid_gelu", "tiny_fused_gelu", "tiny_linear", "merv_full_b1"])
def test_backward_matches_reference_autograd(name, dtype, tol, fused_training):
    # fused_training: the fused forward + _FusedLinearFn backward (no per-encoder projections or their gradients in HBM)
    case = C.CASES[name]
    if dtype == torch.bfloat16 and any(c % 8 for c in case.dims):
        pytest.skip("bf16 path needs C % 8 == 0")
    if fused_training and case.mlp_type != "linear":
        pytest.skip("the fused backward covers the shipped linear projectors")
    if name == "merv_full_b1" and not fused_training:
        pytest.skip("full-size case: fused training path only (the fp64 reference autograd of it is the slow part)")
    g, feats, pp, fp = regenerate(case)
    rng = np.random.default_rng(5)
    G = rng.standard_normal((case.batch, case.token_length, case.llm_dim)).astype(np.float32)
    H = rng.standard_normal((case.batch, case.num_encoders)).astype(np.float32)
    if dtype == torch.bfloat16:  # compare like with like: reference gradients at the bf16-rounded operating point
        feats = [_bf16_round(f) for f in feats]
        pp = [{k: _bf16_round(v) for k, v in p.items()} for p in pp]
        fp = {k: _bf16_round(v) for k, v in fp.items()}
    want_p, want_f = _reference_grads(case, feats, pp, fp, G, H)

    import merv_b200 as M

    m = M.MervFusion.build(case.dims, case.llm_dim, case.out_frames, case.out_size**2, case.mlp_type, text_embedding_dim=case.embed_dim, fused=True)
    m.feature_fusion.fused_training = fused_training  # forced on / off (the default, None, picks the fused path whenever it applies)
    for proj, p in zip(m.projectors, pp):
        proj.projector.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    m.feature_fusion.load_state_dict({k: torch.from_numpy(v) for k, v in fp.items()})
    m = m.to(device=DEV, dtype=dtype).train()
    out, w = m([_t(f, dtype) for f in feats])  # grad mode: module-by-module path through the autograd Functions (or the fused one)
    assert out.requires_grad and w.requires_grad
    assert type(out.grad_fn).__name__.startswith("_FusedLinearFn") == fused_training
    loss = (out.float() * _t(G)).sum() + (w.float() * _t(H)).sum()
    loss.backward()
    for i, proj in enumerate(m.projectors):
        got = dict(proj.projector.named_parameters())  # keys as in the reference state dict: projector[.k].{weight,bias}
        assert sorted(got) == sorted(want_p[i])
        for k, wg in want_p[i].items():
            assert got[k].grad is not None, f"no gradient for projector {i} {k}"
            assert O.rel_err(_np(got[k].grad), wg) < tol, f"gradient of projector {i} {k}"
    ff = m.feature_fusion
    E = case.embed_dim
    assert O.rel_err(_np(ff.Q.grad), want_f["Q"]) < tol
    assert O.rel_err(_np(ff.attention.q_proj_weight.grad), want_f["attention.q_proj_weight"]) < tol
    assert O.rel_err(_np(ff.attention.k_proj_weight.grad), want_f["attention.k_proj_weight"]) < tol
    got_b, want_b = _np(ff.attention.in_proj_bias.grad), want_f["attention.in_proj_bias"]
    assert O.rel_err(got_b[:E], want_b[:E]) < tol
    assert np.abs(want_b[E:]).max() < 1e-6 * np.abs(want_b[:E]).max() and np.abs(got_b[E:]).max() == 0.0  # b_k cancels, b_v is dead
    # exactly like the reference: the discarded attention output leaves v_proj / out_proj without gradient
    assert want_f["attention.v_proj_weight"] is None and ff.attention.v_proj_weight.grad is None
    assert ff.attention.out_proj.weight.grad is None


def test_backward_unsupported_cases_raise():
    import merv_b200 as M

    p = M.AveragePooling3DProjector(64, 128, 4, 4, "linear").to(DEV)
    with pytest.raises(NotImplementedError, match="frozen backbones"):
        p(torch.zeros(1, 4, 16, 64, device=DEV, requires_grad=True))


# ---------------------------------------------------------------------------------------------------------
# boundary contract: stream-ordered, no host sync -> CUDA-graph capturable (SURVEY.md §8b "Threading / streams")
# ---------------------------------------------------------------------------------------------------------
def test_fused_forward_is_cuda_graph_capturable():
    case = C.CASES["mid_linear"]
    g, feats, pp, fp = regenerate(case)
    m = build_module(case, pp, fp, torch.bfloat16, fused=True)
    xs = [_t(f, torch.bfloat16) for f in feats]
    with torch.inference_mode():
        want, want_w = m(xs)  # also builds the cached plan and the input-independent vectors outside the capture
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            m(xs)  # warm the plan for this stream
            with torch.cuda.graph(graph, stream=side):
                out, w = m(xs)
        torch.cuda.synchronize()
        out.zero_()
        for x, f in zip(xs, feats):  # new inputs in the captured buffers, then replay
            x.copy_(_t(f[::-1].copy(), torch.bfloat16))
        graph.replay()
        torch.cuda.synchronize()
        want2, _ = m([_t(f[::-1].copy(), torch.bfloat16) for f in feats])
    assert torch.equal(out, want2), "graph replay must recompute from the captured input buffers"
    assert not torch.equal(want, want2)


def test_misaligned_parameter_views_are_handled():
    # FSDP's use_orig_params=True (fsdp.py:240) hands out parameter views at arbitrary element offsets of a flat buffer
    import merv_b200 as M

    p = M.AveragePooling3DProjector(64, 128, 4, 4, "linear").to(device=DEV, dtype=torch.bfloat16).eval().requires_grad_(False)
    lin = p.projector.projector
    flat = torch.zeros(lin.weight.numel() + 3, device=DEV, dtype=torch.bfloat16)
    flat[3:].copy_(lin.weight.reshape(-1))
    x = torch.randn(2, 4, 16, 64, device=DEV).to(torch.bfloat16)
    with torch.inference_mode():
        want = p(x)
        lin.weight.data = flat[3:].view_as(lin.weight)  # 6-byte offset: not 16-byte aligned
        assert lin.weight.data_ptr() % 16 != 0
        got = p(x)
    assert torch.equal(got, want)


def test_empty_batch_and_more_than_four_encoders():
    import merv_b200 as M

    # (a) an empty batch flows through both paths (a rank that owns no videos, merv_b200/parallel.py)
    case = C.CASES["tiny_linear"]
    g, feats, pp, fp = regenerate(case)
    for fused in (True, False):
        m = build_module(case, pp, fp, torch.bfloat16, fused=fused)
        with torch.inference_mode():
            out, w = m([_t(f[:0], torch.bfloat16) for f in feats])
        assert out.shape == (0, case.token_length, case.llm_dim) and w.shape == (0, case.num_encoders)
    # (b) five encoders: beyond the 4 K-segments of the fused GEMM -> the linked module falls back to the module-by-module
    #     kernels (still sm_100a code, never torch) and must agree with the oracle
    rng = np.random.default_rng(21)
    dims, T, S, K, Eb = (64, 64, 48, 48, 32), 4, 4, 128, 96
    feats5 = [rng.standard_normal((2, T, 16, c), dtype=np.float32) + 0.1 * i for i, c in enumerate(dims)]
    pp5 = [{"projector.weight": rng.uniform(-0.1, 0.1, (K, c)).astype(np.float32), "projector.bias": rng.uniform(-0.1, 0.1, K).astype(np.float32)} for c in dims]
    fp5 = C.make_fusion_params(C.Case("five", 2, (T,) * 5, (16,) * 5, dims, K, Eb, (T,) * 5, S))
    projs = [M.AveragePooling3DProjector(c, K, T, S, "linear") for c in dims]
    ff = M.CrossAttentionAdapterLearnableQuery(Eb, K, T * S * S, averagetoken=True, num_encoder=5)
    m5 = M.MervFusion(projs, ff, fused=True)
    for proj, p in zip(m5.projectors, pp5):
        proj.projector.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    ff.load_state_dict({k: torch.from_numpy(v) for k, v in fp5.items()})
    m5 = m5.to(device=DEV, dtype=torch.float32).eval().requires_grad_(False)
    with torch.inference_mode():
        out, w = m5([_t(f) for f in feats5])
    want, want_w, _ = O.merv_fusion_forward(feats5, pp5, fp5, (T,) * 5, S, "linear", T * S * S)
    assert O.rel_err(_np(out), want) < FP32_TOL and np.abs(_np(w) - want_w).max() < 2e-5


def test_backbone_output_layouts_are_read_in_place():
    # SURVEY.md §8 f-3: the backbones' native outputs are strided views, not fresh tensors:
    #   LanguageBind  [B, 16, 257, C] with a CLS token in front of every frame  (languagebind/__init__.py:85-101)
    #   ViViT         [B, 1 + 16*196, C] with one leading CLS token             (vivit.py:105-114)
    # both must flow through the fused path without a copy and give the same result as their contiguous twins
    import merv_b200 as M

    m = M.MervFusion.build([64, 48], 128, [4, 4], 16, "linear", text_embedding_dim=96, seed=3).to(device=DEV, dtype=torch.bfloat16).eval().requires_grad_(False)
    g = torch.Generator(device=DEV).manual_seed(2)
    lb_full = torch.randn((3, 4, 17, 64), generator=g, device=DEV).to(torch.bfloat16)       # 16 patches + CLS per frame
    vv_full = torch.randn((3, 1 + 4 * 49, 48), generator=g, device=DEV).to(torch.bfloat16)  # CLS + 4 frames x 49 patches
    lb = lb_full[:, :, 1:, :]
    vv = vv_full[:, 1:, :].reshape(3, 4, 49, 48)  # merv.py:576-585 reshape: still a view
    assert not lb.is_contiguous() and not vv.is_contiguous() and vv.data_ptr() == vv_full.data_ptr() + 48 * 2
    with torch.inference_mode():
        out_v, w_v = m([lb, vv])
        out_c, w_c = m([lb.contiguous(), vv.contiguous()])
    assert torch.equal(out_v, out_c) and torch.equal(w_v, w_c)


# ---------------------------------------------------------------------------------------------------------
# host-buffer entry point (what bench.py times as e2e): chunked copy/compute/copy pipeline == one device call
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch", [1, 5, 23])
def test_host_pipeline_matches_device_call(batch):
    from merv_b200.pipeline import HostPipeline

    case = C.CASES["mid_linear"]
    g, feats, pp, fp = regenerate(case)
    m = build_module(case, pp, fp, torch.bfloat16, fused=True)
    reps = -(-batch // case.batch)
    host = [torch.cat([torch.from_numpy(np.ascontiguousarray(f)).to(torch.bfloat16)] * reps)[:batch].contiguous().pin_memory() for f in feats]
    with torch.inference_mode():
        want, want_w = m([h.to(DEV) for h in host])
    pipe = HostPipeline(m, chunk_videos=4)  # 23 videos -> ramp-up, full chunks, ragged chunk, ramp-down
    got, got_w = pipe(host)
    assert got.device.type == "cpu" and got.shape == (batch, case.token_length, case.llm_dim)
    assert torch.equal(got, want.cpu()) and torch.equal(got_w, want_w.cpu())
    got2, _ = pipe(host)  # staging buffers are reused across calls
    assert torch.equal(got2, got)


# ---------------------------------------------------------------------------------------------------------
# SURVEY.md §8 f-4: concat_channel as one K-segmented GEMM == the reference's concat + Linear
# ---------------------------------------------------------------------------------------------------------
def test_concat_channel_segmented_gemm_equals_concat_then_linear():
    from merv_b200 import ops

    torch.manual_seed(3)
    M_, K_, N_ = 640, 256, 512
    Ys = [torch.randn(M_, K_, device=DEV).to(torch.bfloat16) for _ in range(4)]
    W = (torch.randn(N_, 4 * K_, device=DEV) / 32).to(torch.bfloat16)
    b = torch.randn(N_, device=DEV).to(torch.bfloat16)
    got = ops.concat_linear(Ys, W, b)
    want, _ = ops.linear_bias_act(torch.cat(Ys, -1), W, b, 0)  # the plain GEMM on the materialised concatenation
    ref = torch.cat(Ys, -1).float() @ W.float().T + b.float()
    scale = float(ref.abs().max())
    # per-segment TMEM accumulators summed in fp32 registers vs one accumulator: same values up to fp32 summation order
    assert float((got.float() - want.float()).abs().max()) / scale < 1e-2 and float((got.float() - ref).abs().max()) / scale < 5e-3
    mod = __import__("merv_b200").ConcatChannelFusion(4, N_).to(DEV, torch.bfloat16).eval().requires_grad_(False)
    assert sorted(mod.state_dict()) == ["projector.bias", "projector.weight"]  # the reference LinearProjector's keys
    V = [torch.randn(2, 128, N_, device=DEV).to(torch.bfloat16) for _ in range(4)]
    with torch.inference_mode():
        a_, b_ = mod(V), mod(torch.cat(V, -1))  # list call (segmented GEMM) vs the reference's tensor call (plain GEMM)
    assert a_.shape == b_.shape == (2, 128, N_) and float((a_.float() - b_.float()).abs().max()) / float(b_.float().abs().max()) < 1e-2


# ---------------------------------------------------------------------------------------------------------
# SURVEY.md §8 f-2: the whole embedding / mask / label assembly of MERV.forward (merv.py:622-720), unimodal rows included
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mm", [[0, 1, 2, 3, 4], [3, 0], [4]])
def test_forward_multimodal_assembly_matches_oracle(mm):
    case = C.CASES["mid_linear"]
    g, feats, pp, fp = regenerate(case)
    m = build_module(case, pp, fp, torch.bfloat16, fused=True)
    T, K, Bt, L = case.token_length, case.llm_dim, 5, 7
    rep = [torch.cat([_t(f, torch.bfloat16)] * 3)[:Bt].contiguous() for f in feats]  # backbone outputs for the whole batch of 5
    gen = torch.Generator(device="cpu").manual_seed(11)
    emb = torch.randn(Bt, L, K, generator=gen).to(torch.bfloat16).to(DEV)
    mask = (torch.rand(Bt, L, generator=gen) > 0.2).to(DEV)
    labels = torch.randint(0, 32000, (Bt, L), generator=gen).to(DEV)
    labels[:, 0] = -100
    idx = torch.tensor(mm, device=DEV)
    with torch.inference_mode():
        prefix, w0 = m([f[idx] for f in rep])
        whole = len(mm) == Bt
        fe, fm, fl, w = m.forward_multimodal(rep, emb, mask, labels, multimodal_indices=None if whole else idx, bos_token_length=1)
    want_e, want_m, want_l = O.assemble_multimodal(_np(prefix), _np(emb), mask.cpu().numpy(), labels.cpu().numpy(), mm, 1)
    assert fe.shape == (Bt, L + T, K) and fm.dtype == mask.dtype and fl.dtype == labels.dtype
    assert np.array_equal(_np(fe), want_e) and np.array_equal(fm.cpu().numpy(), want_m) and np.array_equal(fl.cpu().numpy(), want_l)
    assert torch.equal(w, w0)
    # no masks / labels given -> None, embeddings unchanged
    with torch.inference_mode():
        fe2, fm2, fl2, _ = m.forward_multimodal(rep, emb, multimodal_indices=None if whole else idx)
    assert fm2 is None and fl2 is None and torch.equal(fe2, fe)


# ---------------------------------------------------------------------------------------------------------
# configuration variants (SURVEY.md §8 f-4): pre_proj_layernorm, concat_channel_ln, averagetoken=False, positional embedding,
# "first" / "concat" — goldens recorded from the unmodified reference modules (tests/golden/variants.npz)
# ---------------------------------------------------------------------------------------------------------
def _variant_names():
    from oracle import variants as V

    return list(V.VARIANTS)


@pytest.mark.parametrize("name", _variant_names())
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_variants_match_reference(name, dtype):
    from tests.variant_util import build_variant_module, run_variant

    mod, v, inputs, gold = build_variant_module(name, dtype, DEV)
    with torch.inference_mode():
        out, w = run_variant(mod, v, inputs, dtype, DEV)
    torch.cuda.synchronize()
    assert tuple(out.shape) == gold["out"].shape and out.dtype == dtype and out.is_contiguous()
    if dtype == torch.float32:
        assert O.rel_err(_np(out), gold["out"]) < FP32_TOL
        if w is not None:
            assert np.abs(_np(w) - gold["weights"]).max() < 2e-5
    else:
        assert O.rel_err(_np(out), gold["out"]) < BF16_TOL
        # the reference's own bf16 run; for the attentive pooler that run alone is 1.0-1.2e-2 away from its fp32 result (bf16 scores
        # and probabilities inside SDPA), so two independent bf16 evaluations get 1.5x the bound between them
        assert O.rel_err(_np(out), gold["out_bf16"]) < (1.5 * BF16_TOL if v["kind"] == "attntv" else BF16_TOL)
        if w is not None:
            assert np.abs(_np(w) - gold["weights"]).max() < 2e-2


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("widths", [[64], [128, 64, 192], [1024, 1024, 768, 768], [4096] * 4])
def test_layernorm_kernel_matches_oracle_incl_segments(widths, dtype):
    # warp-per-row (<= 256 vectors) and CTA-per-row layouts, one and several row segments, strided segment rows
    from merv_b200 import ops

    rng = np.random.default_rng(len(widths) * 1000 + widths[0])
    M_ = 37
    total = sum(widths)
    segs = [rng.standard_normal((M_, k), dtype=np.float32) * (1.0 + 0.5 * i) + 0.3 * i for i, k in enumerate(widths)]
    gamma = (1.0 + 0.3 * rng.standard_normal(total)).astype(np.float32)
    beta = (0.2 * rng.standard_normal(total)).astype(np.float32)
    xs = [_t(s, dtype) for s in segs]
    if len(xs) > 1:  # segment 1 as a column slice of a wider buffer: row stride > width
        wide = torch.zeros((M_, widths[1] + 16), dtype=dtype, device=DEV)
        wide[:, :widths[1]] = xs[1]
        xs[1] = wide[:, :widths[1]]
    y = ops.layernorm(xs, _t(gamma, dtype), _t(beta, dtype), 1e-5)
    torch.cuda.synchronize()
    want = O.layer_norm(np.concatenate([_np(_t(s, dtype)).astype(np.float64) for s in segs], -1), _np(_t(gamma, dtype)).astype(np.float64),
                        _np(_t(beta, dtype)).astype(np.float64))
    assert y.shape == (M_, total) and y.dtype == dtype
    assert O.rel_err(_np(y), want) < (FP32_TOL if dtype == torch.float32 else 6e-3)
    y0 = ops.layernorm(xs, None, None, 1e-5)  # elementwise_affine=False form
    want0 = O.layer_norm(np.concatenate([_np(_t(s, dtype)).astype(np.float64) for s in segs], -1), np.ones(total), np.zeros(total))
    assert O.rel_err(_np(y0), want0) < (FP32_TOL if dtype == torch.float32 else 6e-3)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 2e-5), (torch.bfloat16, 2e-2)])
@pytest.mark.parametrize("widths", [[96], [1024, 512], [4096] * 4])
def test_layernorm_backward_kernel_matches_autograd(widths, dtype, tol):
    from merv_b200 import ops

    rng = np.random.default_rng(17 + len(widths))
    M_, total = 29, sum(widths)
    segs = [_t(rng.standard_normal((M_, k), dtype=np.float32) + 0.2 * i, dtype) for i, k in enumerate(widths)]
    gamma = _t((1.0 + 0.3 * rng.standard_normal(total)).astype(np.float32), dtype)
    dy = _t(rng.standard_normal((M_, total), dtype=np.float32), dtype)
    dx, dg, db = ops.layernorm_backward(segs, dy, gamma, 1e-5)
    torch.cuda.synchronize()
    x64 = torch.cat([s.double() for s in segs], -1).cpu().requires_grad_(True)
    g64 = gamma.double().cpu().requires_grad_(True)
    b64 = torch.zeros(total, dtype=torch.float64, requires_grad=True)
    torch.nn.functional.layer_norm(x64, (total,), g64, b64, 1e-5).backward(dy.double().cpu())
    assert O.rel_err(_np(dx), x64.grad.numpy()) < tol
    assert O.rel_err(_np(dg), g64.grad.numpy()) < tol
    assert O.rel_err(_np(db), b64.grad.numpy()) < tol


@pytest.mark.parametrize("name", ["pre_ln_linear", "pre_ln_gelu", "pre_ln_fused_gelu", "pre_ln_linear_wide"])
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 2e-4), (torch.bfloat16, 3e-2)])
def test_pre_layernorm_projector_backward(name, dtype, tol):
    from tests.variant_util import build_variant_module

    mod, v, inputs, _ = build_variant_module(name, dtype, DEV)
    if dtype == torch.bfloat16 and v["vision_dim"] % 8:
        pytest.skip("bf16 path needs C % 8 == 0")
    mod.requires_grad_(True).train()
    x = _t(inputs[0], dtype)
    rng = np.random.default_rng(3)
    y = mod(x)
    dy = _t(rng.standard_normal(tuple(y.shape), dtype=np.float32), dtype)
    y.backward(dy)
    got = {k: _np(p.grad) for k, p in mod.named_parameters()}
    # fp64 autograd through the same op sequence at the same (rounded) operating point
    ln = torch.nn.LayerNorm(v["vision_dim"]).double()
    ln.load_state_dict({k: t.double().cpu() for k, t in mod.layernorm.state_dict().items()})
    import copy

    seq = copy.deepcopy(mod.projector).cpu().double()
    for p in list(ln.parameters()) + list(seq.parameters()):
        p.grad = None
    seq(ln(x.double().cpu())).backward(dy.double().cpu())
    want = {**{"layernorm." + k: p.grad.numpy() for k, p in ln.named_parameters()}, **{"projector." + k: p.grad.numpy() for k, p in seq.named_parameters()}}
    assert sorted(got) == sorted(want)
    for k in want:
        assert O.rel_err(got[k], want[k]) < tol, k


def test_first_and_token_concat_fusions_on_gpu():
    import merv_b200 as M

    case = C.CASES["mid_linear"]  # 256 tokens per encoder: the direct (batch-strided TMA store) form of "concat"
    g, feats, pp, fp = regenerate(case)
    projs = [M.AveragePooling3DProjector(c, case.llm_dim, t, case.out_size, case.mlp_type) for c, t in zip(case.dims, case.out_frames)]
    for proj, p in zip(projs, pp):
        proj.projector.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
    want = [O.avgpool3d_projector_forward(_bf16_round(f).astype(np.float64), {k: _bf16_round(a).astype(np.float64) for k, a in p.items()}, t,
                                          case.out_size, case.mlp_type) for f, p, t in zip(feats, pp, case.out_frames)]
    for dtype, tol in ((torch.bfloat16, 8e-3), (torch.float32, 8e-3)):
        xs = [_t(f, dtype) for f in feats]
        first = M.MervFusion(projs, None, fusion_type="first").to(device=DEV, dtype=dtype).eval().requires_grad_(False)
        cat = M.MervFusion(projs, None, fusion_type="concat").to(device=DEV, dtype=dtype).eval().requires_grad_(False)
        with torch.inference_mode():
            o1, w1 = first(xs)
            o2, w2 = cat(xs)
        assert w1 is None and w2 is None and o2.shape == (case.batch, case.token_length * case.num_encoders, case.llm_dim)
        assert O.rel_err(_np(o1), want[0]) < tol
        assert O.rel_err(_np(o2), O.token_concat_forward(want)) < tol
        if dtype == torch.bfloat16:  # direct stores must equal "project, then copy into place" bit for bit
            ys = [p._forward_unfused(x) for p, x in zip(first.projectors, xs)]
            assert torch.equal(o2, torch.cat(ys, 1))


def test_positional_embedding_linked_equals_unlinked_on_gpu():
    import merv_b200 as M

    case = C.CASES["mid_linear"]
    g, feats, pp, fp = regenerate(case)
    res = []
    for fused in (False, True):
        projs = [M.AveragePooling3DProjector(c, case.llm_dim, t, case.out_size, case.mlp_type) for c, t in zip(case.dims, case.out_frames)]
        ff = M.CrossAttentionAdapterLearnableQuery(case.embed_dim, case.llm_dim, case.token_length, averagetoken=True,
                                                   num_encoder=case.num_encoders, positional_embedding=True)
        m = M.MervFusion(projs, ff, fused=fused)
        for proj, p in zip(m.projectors, pp):
            proj.projector.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
        ff.load_state_dict({k: torch.from_numpy(v) for k, v in fp.items()}, strict=False)
        with torch.no_grad():
            gen = torch.Generator().manual_seed(9)
            ff.pe.copy_(torch.randn(ff.pe.shape, generator=gen) * 0.5)
        m = m.to(device=DEV, dtype=torch.bfloat16).eval().requires_grad_(False)
        with torch.inference_mode():
            res.append(m([_t(f, torch.bfloat16) for f in feats]))
        pe = _np(ff.pe)
    (o0, w0), (o1, w1) = res
    assert np.abs(_np(w0) - _np(w1)).max() < 1e-2 and O.rel_err(_np(o1), _np(o0)) < 8e-3
    # and against the oracle with the positional embedding (fp64 on the rounded operating point)
    fpr = {k: _bf16_round(v).astype(np.float64) for k, v in fp.items()}
    fpr["pe"] = pe.astype(np.float64)
    ys = [O.avgpool3d_projector_forward(_bf16_round(f).astype(np.float64), {k: _bf16_round(a).astype(np.float64) for k, a in p.items()}, t,
                                        case.out_size, case.mlp_type) for f, p, t in zip(feats, pp, case.out_frames)]
    want, want_w = O.cross_attention_fusion_forward(ys, fpr, case.token_length)
    assert np.abs(_np(w1) - want_w).max() < 1e-2 and O.rel_err(_np(o1), want) < 8e-3
    no_pe = {k: a for k, a in fpr.items() if k != "pe"}
    assert np.abs(O.cross_attention_fusion_forward(ys, no_pe, case.token_length)[1] - want_w).max() > 0.02, "pe must matter in this fixture"


# ---------------------------------------------------------------------------------------------------------
# pieces of the fused backward (include/merv_fusion.h: merv_video_colsum / merv_pair_dot / merv_transpose_rowscale / merv_fused_backward)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_fused_backward_helper_kernels(dtype):
    from merv_b200 import ops

    rng = np.random.default_rng(11)
    B, T, K = 3, 77, 200
    x = _t(rng.standard_normal((B, T, K), dtype=np.float32), dtype)
    y = _t(rng.standard_normal((B, T, K), dtype=np.float32), dtype)
    cs = ops.video_colsum(x, 0.5)
    assert cs.shape == (B, K) and cs.dtype == torch.float32
    assert O.rel_err(_np(cs), _np(x).astype(np.float64).sum(1) * 0.5) < 1e-5
    xs = x[:, 5:, :]  # strided videos (batch stride > T * K)
    assert O.rel_err(_np(ops.video_colsum(xs)), _np(xs).astype(np.float64).sum(1)) < 1e-5
    pd = ops.pair_dot(x, y)
    want = (_np(x).astype(np.float64) * _np(y).astype(np.float64)).reshape(B, -1).sum(1)
    assert np.abs(_np(pd).astype(np.float64).sum(1) - want).max() < 1e-4 * np.abs(want).max() + 1e-3
    # transpose with per-video row scale and zero-filled padding columns
    R, Cc, rows = 77 * 3, 200, 77
    m2 = x.reshape(R, Cc)
    sc = _t(rng.standard_normal((B, 4), dtype=np.float32))[:, 2]  # strided scale column, like weights[:, e]
    yt = ops.transpose(m2, pad=True, row_scale=sc, rows_per_scale=rows)
    vec = 8 if dtype == torch.bfloat16 else 4
    Rp = -(-R // vec) * vec
    assert yt.shape == (Cc, Rp)
    want_t = (_np(m2) * np.repeat(_np(sc), rows)[:, None]).T
    assert O.rel_err(_np(yt[:, :R]), want_t) < (1e-6 if dtype == torch.float32 else 4e-3)
    assert Rp == R or float(yt[:, R:].abs().max()) == 0.0
    yt2 = ops.transpose(m2, pad=True)
    assert torch.equal(yt2[:, :R], m2.T) and (Rp == R or float(yt2[:, R:].abs().max()) == 0.0)


def test_fused_training_matches_module_by_module_training():
    # same parameters, same inputs: the two training paths must produce the same outputs and (to bf16 accuracy) the same gradients
    import merv_b200 as M

    case = C.CASES["mid_linear"]
    g, feats, pp, fp = regenerate(case)
    rng = np.random.default_rng(2)
    G = _t(rng.standard_normal((case.batch, case.token_length, case.llm_dim), dtype=np.float32))
    H = _t(rng.standard_normal((case.batch, case.num_encoders), dtype=np.float32))
    grads = []
    for fused_training in (False, True):
        m = M.MervFusion.build(case.dims, case.llm_dim, case.out_frames, case.out_size**2, case.mlp_type, text_embedding_dim=case.embed_dim, fused=True)
        m.feature_fusion.fused_training = fused_training
        for proj, p in zip(m.projectors, pp):
            proj.projector.load_state_dict({k: torch.from_numpy(v) for k, v in p.items()})
        m.feature_fusion.load_state_dict({k: torch.from_numpy(v) for k, v in fp.items()})
        m = m.to(device=DEV).train()  # fp32 master weights, bf16 autocast: the training configuration (base_strategy.py:210-214)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out, w = m([_t(f, torch.bfloat16) for f in feats])
        assert out.dtype == torch.bfloat16
        ((out.float() * G).sum() + (w.float() * H).sum()).backward()
        grads.append(({k: _np(p.grad) for k, p in m.named_parameters() if p.grad is not None}, _np(out), _np(w)))
        assert all(p.grad.dtype == torch.float32 for p in m.parameters() if p.grad is not None)
    (g0, o0, w0), (g1, o1, w1) = grads
    assert sorted(g0) == sorted(g1)
    assert O.rel_err(o1, o0) < 8e-3 and np.abs(w1 - w0).max() < 1e-2
    for k in g0:
        assert O.rel_err(g1[k], g0[k]) < 3e-2, k


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("N,K", [(4096, 1024), (512, 768), (384, 4096), (100, 72)])
def test_affine_score_vec_two_stage_gemv(N, K, dtype):
    # v = W^T u, c = u . b: the narrow shapes take the two-stage transposed GEMV, (100, 72) the single-stage kernel's tail handling
    from merv_b200 import ops

    rng = np.random.default_rng(N + K)
    W = _t(rng.standard_normal((N, K), dtype=np.float32) / np.sqrt(N), dtype)
    b = _t(rng.standard_normal(N, dtype=np.float32), dtype)
    u = _t(rng.standard_normal(N, dtype=np.float32))
    v, c = ops.affine_score_vec(W, b, u)
    want_v = _np(W).astype(np.float64).T @ _np(u).astype(np.float64)
    assert O.rel_err(_np(v), want_v) < 1e-5
    assert abs(float(c) - float(_np(b).astype(np.float64) @ _np(u).astype(np.float64))) < 1e-4 * max(1.0, abs(float(c)))
    v2, _ = ops.affine_score_vec(W, b, u)
    assert torch.equal(v, v2)  # fixed summation order


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("heads,hd,n_q,n_kv,batches,shared_q", [(8, 128, 64, 256, 3, True), (8, 96, 64, 196, 2, True), (4, 8, 5, 9, 2, False),
                                                                  (2, 32, 37, 70, 1, True), (8, 128, 64, 256, 40, True), (3, 64, 128, 200, 5, False)])
@pytest.mark.parametrize("impl", ["tcgen05", "simt"])
def test_cross_attention_kernel_matches_oracle(heads, hd, n_q, n_kv, batches, shared_q, dtype, impl, monkeypatch):
    # head dims 128 / 96 / 32 / 8, ragged query and key counts (tails of the 32-query pass and of the key chunks), shared and per-entry queries.
    # bf16 with head_dim % 32 == 0 runs both contractions on the tensor cores (attention_tcgen05.cu: S = Q K^T and O = P V as tcgen05.mma,
    # P rounded to bf16 in between, as in flash attention); impl == "simt" forces the CUDA-core kernel for the same inputs.
    from merv_b200 import ops

    if impl == "simt":
        monkeypatch.setenv("MERV_ATTN_IMPL", "simt")
    elif dtype != torch.bfloat16 or hd % 32:
        pytest.skip("the tcgen05 kernel covers bf16 with head_dim % 32 == 0")
    rng = np.random.default_rng(heads * 1000 + hd)
    C_ = heads * hd
    q = _t(rng.standard_normal((n_q, C_) if shared_q else (batches, n_q, C_), dtype=np.float32), dtype)
    kv = _t(rng.standard_normal((batches * n_kv, 2 * C_), dtype=np.float32), dtype)
    out = ops.cross_attention(q, kv, batches, heads)
    torch.cuda.synchronize()
    qf = _np(q).astype(np.float64)
    qf = np.broadcast_to(qf, (batches, n_q, C_)) if shared_q else qf
    kvf = _np(kv).astype(np.float64).reshape(batches, n_kv, 2, heads, hd)
    k, v = kvf[:, :, 0].transpose(0, 2, 1, 3), kvf[:, :, 1].transpose(0, 2, 1, 3)
    qh = qf.reshape(batches, n_q, heads, hd).transpose(0, 2, 1, 3)
    att = O._softmax_last((qh @ k.transpose(0, 1, 3, 2)) * hd ** -0.5)
    want = (att @ v).transpose(0, 2, 1, 3).reshape(batches, n_q, C_)
    assert out.shape == want.shape and out.dtype == dtype
    assert O.rel_err(_np(out), want) < (FP32_TOL if dtype == torch.float32 else (1e-2 if impl == "tcgen05" else 6e-3))
    a = _t(rng.standard_normal((batches * n_q, C_), dtype=np.float32), dtype)
    b = _t(rng.standard_normal((n_q, C_), dtype=np.float32), dtype)
    got = ops.add_rows(a, b)
    want_add = (_np(a).reshape(batches, n_q, C_) + _np(b)).reshape(batches * n_q, C_)
    assert O.rel_err(_np(got), want_add) < (1e-6 if dtype == torch.float32 else 4e-3)


@pytest.mark.parametrize("heads,hd,n_q,n_kv,batches,shared_q", [(8, 128, 64, 256, 3, True), (8, 96, 64, 196, 2, True), (2, 32, 37, 70, 1, True),
                                                                  (3, 64, 64, 200, 5, False), (8, 128, 64, 256, 37, True)])
def test_cross_attention_backward_kernel_matches_autograd(heads, hd, n_q, n_kv, batches, shared_q):
    """merv_cross_attention_backward (five tcgen05 contractions per frame and head; S / P recomputed) against fp64 autograd through the
    attention of CrossAttention.forward (nn_utils.py:393-412) on the same bf16-rounded inputs."""
    from merv_b200 import ops

    rng = np.random.default_rng(heads * 100 + hd + n_kv)
    C_ = heads * hd
    q = _t(rng.standard_normal((n_q, C_) if shared_q else (batches, n_q, C_), dtype=np.float32), torch.bfloat16)
    kv = _t(rng.standard_normal((batches * n_kv, 2 * C_), dtype=np.float32), torch.bfloat16)
    dout = _t(rng.standard_normal((batches, n_q, C_), dtype=np.float32), torch.bfloat16)
    dq, dkv = ops.cross_attention_backward(q, kv, dout, batches, heads)
    torch.cuda.synchronize()
    qq = (q.double().unsqueeze(0).expand(batches, n_q, C_) if shared_q else q.double()).clone().requires_grad_(True)
    kk = kv.double().clone().requires_grad_(True)
    k5 = kk.view(batches, n_kv, 2, heads, hd)
    qh = qq.view(batches, n_q, heads, hd).permute(0, 2, 1, 3)
    att = torch.softmax(qh @ k5[:, :, 0].permute(0, 2, 3, 1) * hd ** -0.5, -1)
    out = (att @ k5[:, :, 1].permute(0, 2, 1, 3)).permute(0, 2, 1, 3).reshape(batches, n_q, C_)
    want_dq, want_dkv = torch.autograd.grad(out, [qq, kk], dout.double())
    assert dq.shape == (batches, n_q, C_) and dkv.shape == (batches * n_kv, 2 * C_)
    assert O.rel_err(_np(dq), want_dq.cpu().numpy()) < 1.5e-2
    assert O.rel_err(_np(dkv[:, :C_]), want_dkv[:, :C_].cpu().numpy()) < 1.5e-2   # dK
    assert O.rel_err(_np(dkv[:, C_:]), want_dkv[:, C_:].cpu().numpy()) < 1.5e-2   # dV
    dq2, dkv2 = ops.cross_attention_backward(q, kv, dout, batches, heads)
    assert torch.equal(dq, dq2) and torch.equal(dkv, dkv2)  # deterministic


@pytest.mark.parametrize("C_,llm,n,heads,F,N,B,mlp_type", [(256, 128, 16, 8, 3, 49, 2, "gelu-mlp"), (1024, 512, 64, 8, 4, 256, 2, "linear"),
                                                          (768, 256, 64, 8, 2, 196, 1, "linear")])
def test_attentive_pooler_training_matches_reference_autograd(C_, llm, n, heads, F, N, B, mlp_type):
    """Forward + backward of the `attntv` resampler (bf16, attention and every Linear on the tensor cores) against torch autograd through
    the UNMODIFIED reference AttentivePooler in fp32 on the same bf16-rounded parameters (oracle/_ref travels with the snapshot)."""
    import copy

    import merv_b200 as M
    from oracle.ref_loader import load_reference_nn_utils

    ref = load_reference_nn_utils()
    torch.manual_seed(C_ + n)
    r = ref.AttentivePooler(C_, llm, num_query_tokens=n, num_heads=heads, output_frames=F, mlp_type=mlp_type)
    with torch.no_grad():
        for name, p in r.named_parameters():
            if name.endswith("bias") or "norm" in name:
                p.add_(0.1 * torch.randn_like(p))
        r.query_tokens.mul_(20.0)
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
    assert O.rel_err(_np(out), _np(want)) < BF16_TOL
    got = dict(m.named_parameters())
    for name, p in r.named_parameters():
        assert got[name].grad is not None, name
        scale = float(p.grad.abs().max())
        err = float((got[name].grad.float() - p.grad).abs().max())
        assert err <= 4e-2 * scale + 1e-6, (name, err / max(scale, 1e-12))
    with torch.inference_mode():  # and the inference path agrees with the training path's forward
        out_inf = m(x)
    assert O.rel_err(_np(out_inf), _np(out)) < 1e-2


@pytest.mark.parametrize("B,head", [(48, None), (24, 1), (24, 23)])  # None: the library's default head (40 videos)
def test_pool_assist_is_bit_identical_to_the_three_launch_path(B, head, monkeypatch):
    """Pool assist (merv_b200/csrc/pool_assist.cuh, opt-in with MERV_POOL_ASSIST=1): the GEMM's spare warps pool, score and soft-max the
    videos behind the head inside the GEMM launch, handing them to the tensor cores through per-video release / acquire flags.  Same
    arithmetic and summation order as the standalone kernels -> prefix and weights must be BIT-identical, on the plain call, on re-runs
    of the cached plan (the flags are reset by the scores kernel), with the gather by multimodal_indices and with the prefix written
    into a strided slot of the embedding buffer."""
    m = _full_module(True)
    feats = _full_features(B)
    idx = torch.tensor([3, 0, 7, 23, 11, 5, 19, 2, 14, 9, 21, 1, 16, 8, 22, 4, 13, 6], dtype=torch.int32, device=DEV)
    emb = torch.zeros((B, 1 + 1024 + 7, 4096), dtype=torch.bfloat16, device=DEV)
    with torch.inference_mode():
        monkeypatch.setenv("MERV_POOL_ASSIST", "0")
        want, want_w = m(feats)
        want_g, want_gw = m(feats, batch_index=idx)
        torch.cuda.synchronize()
        monkeypatch.setenv("MERV_POOL_ASSIST", "1")
        if head is not None:
            monkeypatch.setenv("MERV_ASSIST_HEAD", str(head))
        for _ in range(3):
            out, w = m(feats)
            assert torch.equal(out, want) and torch.equal(w, want_w)
        out_g, w_g = m(feats, batch_index=idx)
        assert torch.equal(out_g, want_g) and torch.equal(w_g, want_gw)
        m(feats, out=emb[:, 1:1025])
        torch.cuda.synchronize()
        assert torch.equal(emb[:, 1:1025], want) and not emb[:, 0].any() and not emb[:, 1025:].any()


@pytest.mark.parametrize("F,H,T,S,Cc", [(5, 7, 2, 3, 24), (2, 16, 2, 8, 128), (3, 14, 3, 8, 64), (4, 6, 2, 2, 8)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("impl", ["tma", "direct"])
def test_pool3d_displaced_windows_match_oracle(F, H, T, S, Cc, dtype, impl, monkeypatch):
    """merv_pool_desc.shift_*: the 27 displaced poolings of a zero-padded 3 x 3 x 3 convolution (ops.pool3d_conv_taps), TMA kernel (box
    coordinates displaced, out-of-grid zero fill by the TMA unit) and the plain-load kernel, against the oracle's pooling of an explicitly
    zero-padded, displaced copy."""
    from merv_b200 import ops

    if impl == "direct":
        monkeypatch.setenv("MERV_POOL_IMPL", "direct")
    if dtype == torch.bfloat16 and Cc % 8:
        pytest.skip("channel count not a multiple of the 16-byte vector for this dtype")
    rng = np.random.default_rng(F * 100 + H)
    x = _t(rng.standard_normal((2, F, H * H, Cc)).astype(np.float32) + 0.3, dtype)
    A = ops.pool3d_conv_taps(x, T, S)
    torch.cuda.synchronize()
    assert A.shape == (2, T * S * S, 27 * Cc) and A.dtype == dtype
    xn = _np(x).reshape(2, F, H, H, Cc)
    xp = np.zeros((2, F + 2, H + 2, H + 2, Cc), dtype=xn.dtype)
    xp[:, 1:-1, 1:-1, 1:-1] = xn
    tol = 1e-6 if dtype == torch.float32 else 4e-3
    for tap, (sf, sh, sw) in enumerate(ops.CONV_TAPS):
        shifted = xp[:, 1 + sf:1 + sf + F, 1 + sh:1 + sh + H, 1 + sw:1 + sw + H].reshape(2, F, H * H, Cc)
        want = O.avg_pool3d_tokens(shifted, T, S)
        got = _np(A[:, :, tap * Cc:(tap + 1) * Cc])
        assert np.abs(got - want).max() <= tol * max(1.0, np.abs(want).max()), (tap, (sf, sh, sw))


@pytest.mark.parametrize("C_,llm,F,H,T,S,B,mlp_type", [(128, 256, 2, 16, 2, 8, 2, "linear"), (64, 128, 4, 14, 2, 8, 1, "gelu-mlp"), (24, 32, 5, 7, 2, 3, 2, "linear")])
def test_conv3d_projector_training_matches_reference_autograd(C_, llm, F, H, T, S, B, mlp_type):
    """Forward + backward of the `3dconv` resampler in bf16 (27 displaced poolings + ONE tcgen05 GEMM with K = 27 C; dW = dY^T A read
    MN-major in place) against torch autograd through the UNMODIFIED reference Convolutional3DProjector in fp32 on the same bf16-rounded
    parameters — the reference convolves the un-pooled grid and pools afterwards."""
    import copy

    import merv_b200 as M
    from oracle.ref_loader import load_reference_nn_utils

    ref = load_reference_nn_utils()
    torch.manual_seed(C_ + H)
    r = ref.Convolutional3DProjector(C_, llm, output_frames=T, output_size=S, mlp_type=mlp_type)
    m = M.Convolutional3DProjector.from_reference(copy.deepcopy(r)).to(device=DEV, dtype=torch.bfloat16)
    r = r.to(torch.bfloat16).float().to(DEV)
    g = torch.Generator().manual_seed(5)
    x = (torch.randn((B, F, H * H, C_), generator=g) + 0.3).to(torch.bfloat16).to(DEV)
    G = torch.randn((B, T * S * S, llm), generator=g).to(DEV)
    out = m(x)
    out.backward(G.to(torch.bfloat16))
    want = r(x.float())
    want.backward(G)
    torch.cuda.synchronize()
    assert O.rel_err(_np(out), _np(want)) < BF16_TOL
    got = dict(m.named_parameters())
    for name, p in r.named_parameters():
        assert got[name].grad is not None and got[name].grad.shape == p.grad.shape, name
        scale = float(p.grad.abs().max())
        err = float((got[name].grad.float() - p.grad).abs().max())
        assert err <= 4e-2 * scale + 1e-6, (name, err / max(scale, 1e-12))
    with torch.inference_mode():
        out_inf = m(x)
    assert O.rel_err(_np(out_inf), _np(out)) < 1e-2


@pytest.mark.parametrize("videos,T,N_out,Cc", [(3, 64, 256, 128), (2, 128, 136, 200), (5, 192, 384, 776), (4, 1024, 4096, 768)])
@pytest.mark.parametrize("cta_group", [1, 2])
@pytest.mark.parametrize("split", [None, 1, 2, 3])  # None: the library's choice; k: the videos in k ranges, fp32 partial tiles folded afterwards
def test_wgrad_video_matches_fp32_reference(videos, T, N_out, Cc, cta_group, split, monkeypatch):
    """merv_wgrad_video: dW = sum_b scale[b] dY[b]^T X[b] and the per-video <W, dY[b]^T X[b]> from one tcgen05 pass (accumulator drained
    once per video), against fp32 torch on the same bf16 inputs; M / N tails, several k-blocks per video, the merv-full shape."""
    from merv_b200 import ops

    monkeypatch.setenv("MERV_GEMM_CTA_GROUP", str(cta_group))  # single CTA (the default for this kernel) / CTA pair
    if split is not None:
        monkeypatch.setenv("MERV_WGRAD_SPLIT", str(split))
    g = torch.Generator(device=DEV).manual_seed(videos * 1000 + T)
    dy = torch.randn((videos * T, N_out), generator=g, device=DEV).to(torch.bfloat16)
    x = (torch.randn((videos * T, Cc), generator=g, device=DEV) + 0.2).to(torch.bfloat16)
    w = (torch.randn((N_out, Cc), generator=g, device=DEV) * 0.05).to(torch.bfloat16)
    scale_full = torch.rand((videos, 4), generator=g, device=DEV) + 0.1
    scale = scale_full[:, 2]  # strided, as the mixing weights [B, E] of one encoder are
    dW, partial = ops.wgrad_video(dy, x, scale, w, videos)
    dW2, partial2 = ops.wgrad_video(dy, x, scale, w, videos)
    torch.cuda.synchronize()
    assert torch.equal(dW, dW2) and torch.equal(partial, partial2)  # deterministic
    G = torch.einsum("btn,btc->bnc", dy.float().view(videos, T, N_out), x.float().view(videos, T, Cc))
    want_dW = (scale.view(-1, 1, 1) * G).sum(0)
    want_dot = (G * w.float()).sum((1, 2))
    assert dW.shape == (N_out, Cc) and dW.dtype == torch.bfloat16
    assert float((dW.float() - want_dW).abs().max()) <= 6e-3 * float(want_dW.abs().max())  # bf16 rounding of the result
    got_dot = partial.double().sum(1)
    assert float((got_dot - want_dot.double()).abs().max()) <= 2e-4 * max(1.0, float(want_dot.abs().max()))


@pytest.mark.parametrize("arch,fusion", [("3dconv+linear", "cross_attention_avg_lq"), ("3dconv+frame2+gelu-mlp", "concat_channel"),
                                         ("3davg+frame2+linear", "concat_channel_ln"), ("avg+gelu-mlp", "scalar")])
def test_from_config_forward_matches_the_reference_modules(arch, fusion):
    """A whole configuration built from the reference's config strings (MervFusion.from_config, merv.py:87-227) and run on the GPU in bf16,
    against the UNMODIFIED reference modules constructed in MERV.__init__'s order from the same seed and glued as merv.py:587-609 glues
    them, in fp32 on the same bf16-rounded parameters and inputs.  Covers the resamplers / mixers outside the shipped configuration
    end to end (3dconv in front of the learnable-query mixer and of concat_channel, frame factors, the scalar mixer)."""
    import functools
    import re

    import merv_b200 as M
    from oracle.ref_loader import load_reference_nn_utils

    ref = load_reference_nn_utils()
    dims, llm, temporal, ptl, H = [64, 48], 128, [4, 4], 16, 6
    if fusion == "scalar":  # the reference's ScalarAdapter always holds four scalars (nn_utils.py:527): four encoders
        dims, temporal = [64, 48, 32, 40], [4, 4, 4, 4]
    factor = int(re.search(r"frame(\d+)", arch).group(1)) if "frame" in arch else 1
    vfl = (temporal[0] // factor) * ptl
    m = M.MervFusion.from_config(dims, llm, temporal, arch_specifier=arch, feature_fusion=fusion, projector_token_length=ptl, visual_feature_length=vfl)
    torch.manual_seed(dims[0])  # merv.py:87
    mlp_type = "linear" if arch.endswith("linear") else "gelu-mlp"
    parts = arch.split("+")
    P = (functools.partial(ref.Convolutional3DProjector, output_size=4) if "3dconv" in parts else
         functools.partial(ref.AveragePooling3DProjector, output_size=4) if "3davg" in parts else functools.partial(ref.AveragePoolingProjector, output_size=4))
    projs = [P(c, llm, output_frames=t // factor, mlp_type=mlp_type) for c, t in zip(dims, temporal)]
    if fusion == "cross_attention_avg_lq":
        ff = ref.CrossAttentionAdapterLearnableQuery(embed_dim=3072, llm_dim=llm, token_length=vfl, averagetoken=True)
    elif fusion == "concat_channel":
        ff = ref.LinearProjector(len(dims) * llm, llm)
    elif fusion == "concat_channel_ln":
        ff = torch.nn.Sequential(torch.nn.LayerNorm(len(dims) * llm), ref.LinearProjector(len(dims) * llm, llm))
    else:
        ff = ref.ScalarAdapter(len(dims))
    with torch.no_grad():
        if fusion == "cross_attention_avg_lq":  # far from the flat softmax of the default init, identically on both sides
            ff.Q.mul_(64.0)
            m.feature_fusion.Q.mul_(64.0)
        if fusion == "scalar":
            ff.scalar.copy_(torch.tensor([0.7, -0.4, 0.1, 0.3]))
            m.feature_fusion.scalar.copy_(torch.tensor([0.7, -0.4, 0.1, 0.3]))
    m = m.to(device=DEV, dtype=torch.bfloat16).eval().requires_grad_(False)
    refs = torch.nn.ModuleList(projs).to(torch.bfloat16).float().to(DEV).eval()
    ff = ff.to(torch.bfloat16).float().to(DEV).eval()
    g = torch.Generator().manual_seed(3)
    xs = [(torch.randn((2, t, H * H, c), generator=g) + 0.2 * i).to(torch.bfloat16).to(DEV) for i, (c, t) in enumerate(zip(dims, temporal))]
    with torch.inference_mode():
        out, w = m(xs)
        ys = [p(x.float()) for p, x in zip(refs, xs)]
        if fusion in ("concat_channel", "concat_channel_ln"):  # merv.py:603-606
            want, want_w = ff(torch.concat(ys, -1)), None
        elif fusion == "scalar":  # the module's own forward (MERV.forward has no branch for it)
            want, want_w = ff(ys)
        else:  # merv.py:607-609
            want, want_w = ff(ys)
    torch.cuda.synchronize()
    assert tuple(out.shape) == tuple(want.shape) == (2, vfl, llm)
    assert O.rel_err(_np(out), _np(want)) < BF16_TOL
    if want_w is not None:
        assert w is not None and np.abs(_np(w) - _np(want_w)).max() < 2e-2
        if fusion == "cross_attention_avg_lq":
            assert (want_w.max(-1).values - want_w.min(-1).values).mean() > 0.02, "degenerate softmax: the score path would not be exercised"
