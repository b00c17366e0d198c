"""CPU tests: the numpy oracle (oracle/fusion_oracle.py) against fixtures produced by the UNMODIFIED
reference modules (oracle/make_golden.py -> tests/golden/*.npz).  The reference has no tests of its own
(SURVEY.md §4), so these fixtures are what pins the oracle."""
import numpy as np
import pytest

from oracle import cases as C
from oracle import fusion_oracle as O
from tests.golden_util import regenerate

FP32_TOL = 1e-5  # BASELINE.json north_star: 1e-5 relative in fp32 (metric: max|a-b| / max|b|)


def test_window_table_14_to_8():
    # SURVEY.md §7: 14 -> 8 has overlapping windows of size 2/3/3/2/2/3/3/2
    assert O.adaptive_windows(14, 8) == [(0, 2), (1, 4), (3, 6), (5, 7), (7, 9), (8, 11), (10, 13), (12, 14)]
    assert O.adaptive_windows(16, 8) == [(2 * i, 2 * i + 2) for i in range(8)]
    assert O.adaptive_windows(16, 16) == [(i, i + 1) for i in range(16)]
    assert O.adaptive_windows(5, 3) == [(0, 2), (1, 4), (3, 5)]


def test_token_order_is_f_h_w():
    # token index = f*S*S + h*S + w with w fastest (SURVEY.md §8 a2)
    F, H, S, Cc = 2, 4, 2, 3
    x = np.zeros((1, F, H * H, Cc), np.float32)
    for f in range(F):
        for h in range(H):
            for w in range(H):
                x[0, f, h * H + w, :] = 100 * f + 10 * (h // 2) + (w // 2)
    y = O.avg_pool3d_tokens(x, F, S)
    expect = [100 * f + 10 * i + j for f in range(F) for i in range(S) for j in range(S)]
    assert np.allclose(y[0, :, 0], expect)


@pytest.mark.parametrize("name", list(C.CASES))
def test_oracle_matches_reference_golden(name):
    case = C.CASES[name]
    g, feats, pp, fp = regenerate(case)
    out, w, ys = O.merv_fusion_forward(feats, pp, fp, case.out_frames, case.out_size, case.mlp_type, case.token_length)
    assert out.shape == (case.batch, case.token_length, case.llm_dim)
    scale = float(g["out_abs_max"])
    if case.fusion == "concat_channel":  # no mixing weights on this path (merv.py:603-606)
        assert w.shape == (case.batch, 0) and g["weights"].shape == (case.batch, 0)
    else:
        assert w.shape == ((1 if case.fusion == "scalar" else case.batch), case.num_encoders)  # ScalarAdapter returns [1, E]
        assert np.allclose(w.sum(-1), 1.0, atol=1e-5)
        assert np.abs(w - g["weights"]).max() < 2e-5
    idx = g["sample_idx"]
    assert np.abs(out.reshape(-1)[idx] - g["out_samples"]).max() / scale < FP32_TOL
    assert abs(float(out.astype(np.float64).sum()) - float(g["out_sum"])) < 1e-4 * max(1.0, abs(float(g["out_abs_mean"])) * out.size) 
    for e, y in enumerate(ys):
        ref = g["y_samples"][e]
        assert np.abs(y.reshape(-1)[idx % y.size] - ref).max() / max(np.abs(ref).max(), 1e-6) < FP32_TOL
    if name in C.FULL_STORE_CASES:
        assert O.rel_err(out, g["out"]) < FP32_TOL
        for e, x in enumerate(feats):
            pooled = O.avg_pool3d_tokens(x, case.out_frames[e], case.out_size)
            assert O.rel_err(pooled, g[f"pooled{e}"]) < FP32_TOL
            assert O.rel_err(ys[e], g[f"y{e}"]) < FP32_TOL


@pytest.mark.parametrize("name", ["tiny_linear", "ragged_windows", "mid_linear"])
def test_query_vector_identity(name):
    # weights == softmax_e(u . mean_t V_e): the algebra the CUDA score kernels rely on (SURVEY.md §3.3)
    case = C.CASES[name]
    g, feats, pp, fp = regenerate(case)
    _, w, ys = O.merv_fusion_forward(feats, pp, fp, case.out_frames, case.out_size, case.mlp_type, case.token_length)
    u = O.fusion_query_vector(fp)
    s = np.stack([y.astype(np.float64).mean(1) @ u.astype(np.float64) for y in ys], axis=1)
    e = np.exp(s - s.max(-1, keepdims=True))
    assert np.abs(e / e.sum(-1, keepdims=True) - w).max() < 1e-5


def test_single_encoder_is_identity():
    case = C.CASES["single_encoder"]
    g, feats, pp, fp = regenerate(case)
    out, w, ys = O.merv_fusion_forward(feats, pp, fp, case.out_frames, case.out_size, case.mlp_type, case.token_length)
    assert np.array_equal(w, np.ones_like(w))
    assert np.array_equal(out, ys[0])


def test_token_length_one_broadcast():
    # nn_utils.py:502: an encoder emitting a single token is repeated to token_length
    case = C.CASES["tiny_linear"]
    fp = C.make_fusion_params(case)
    rng = np.random.default_rng(0)
    V = [rng.standard_normal((2, case.token_length, case.llm_dim)).astype(np.float32),
         rng.standard_normal((2, 1, case.llm_dim)).astype(np.float32)]
    out, w = O.cross_attention_fusion_forward(V, fp, case.token_length)
    Vb = [V[0], np.repeat(V[1], case.token_length, axis=1)]
    out2, w2 = O.cross_attention_fusion_forward(Vb, fp, case.token_length)
    assert np.array_equal(out, out2) and np.array_equal(w, w2)
    with pytest.raises(AssertionError):
        O.cross_attention_fusion_forward([V[0][:, :3]], fp, case.token_length)


def test_unsupported_projector_type():
    with pytest.raises(ValueError):
        O.projector_forward(np.zeros((1, 4), np.float32), {}, "relu-mlp")


@pytest.mark.parametrize("name", ["tiny_linear", "tiny_gelu", "tiny_fused_gelu", "ragged_windows", "mid_linear"])
def test_torch_port_cpu_baseline_matches_golden(name):
    # the timed CPU baseline (bench.py cpu_baseline / --impl reference) must compute the same thing
    import torch

    from oracle import torch_port

    case = C.CASES[name]
    g, feats, pp, fp = regenerate(case)
    tt = lambda d: {k: torch.from_numpy(v) for k, v in d.items()}  # noqa: E731
    out, w = torch_port.fusion_forward([torch.from_numpy(f) for f in feats], [tt(p) for p in pp], tt(fp), case.out_frames,
                                       case.out_size, case.mlp_type, case.token_length)
    idx = g["sample_idx"]
    assert np.abs(out.numpy().reshape(-1)[idx] - g["out_samples"]).max() / float(g["out_abs_max"]) < FP32_TOL
    assert np.abs(w.numpy() - g["weights"]).max() < 2e-5


def test_assemble_multimodal_layout():
    # merv.py:622-720: [BOS | prefix | text] rows first, then text-only rows padded at the END; prefix positions IGNORE_INDEX / True
    rng = np.random.default_rng(0)
    Bt, L, T, K = 4, 5, 3, 2
    emb = rng.standard_normal((Bt, L, K)).astype(np.float32)
    mask = rng.random((Bt, L)) > 0.3
    labels = rng.integers(0, 100, (Bt, L))
    prefix = rng.standard_normal((2, T, K)).astype(np.float32)
    fe, fm, fl = O.assemble_multimodal(prefix, emb, mask, labels, [2, 0], 1)
    assert fe.shape == (Bt, L + T, K) and fm.shape == fl.shape == (Bt, L + T)
    assert np.array_equal(fe[0, :1], emb[2, :1]) and np.array_equal(fe[0, 1:1 + T], prefix[0]) and np.array_equal(fe[0, 1 + T:], emb[2, 1:])
    assert fm[:2, 1:1 + T].all() and (fl[:2, 1:1 + T] == O.IGNORE_INDEX).all()
    assert np.array_equal(fe[2, :L], emb[1]) and not fe[2:, L:].any()          # unimodal rows 1 and 3, zero padded at the end
    assert not fm[2:, L:].any() and (fl[2:, L:] == O.IGNORE_INDEX).all() and np.array_equal(fl[3, :L], labels[3])
    fe2, fm2, fl2 = O.assemble_multimodal(np.concatenate([prefix, prefix]), emb, mask, labels, [0, 1, 2, 3], 1)
    assert fe2.shape == (Bt, L + T, K)  # no unimodal rows: fused == multimodal


# ---- configuration variants (SURVEY.md §8 f-4): pre_proj_layernorm, concat_channel_ln, averagetoken=False, positional embedding ----
def oracle_variant(v, inputs, params):
    if v["kind"] == "projector":
        return O.projector_forward(inputs[0], params, v["mlp_type"]), None
    if v["kind"] == "attntv":
        return O.attentive_pooler_forward(inputs[0], params, v["heads"], v["mlp_type"]), None
    if v["kind"] == "conv3d":
        return O.conv3d_projector_forward(inputs[0], params, v["T"], v["S"], v["mlp_type"]), None
    if v["kind"] == "concat_channel_ln":
        return O.concat_channel_ln_forward(inputs, params), None
    return O.cross_attention_fusion_forward(inputs, params, v["T"], averagetoken=v["averagetoken"])


def _variant_names():
    from oracle import variants as V

    return list(V.VARIANTS)


@pytest.mark.parametrize("name", _variant_names())
def test_oracle_variants_match_reference_golden(name):
    from tests.golden_util import load_variant

    v, inputs, params, gold = load_variant(name)
    out, w = oracle_variant(v, inputs, params)
    assert out.shape == gold["out"].shape
    assert O.rel_err(out, gold["out"]) < FP32_TOL
    if w is not None:
        assert np.abs(w - gold["weights"]).max() < 2e-5 and np.allclose(w.sum(-1), 1.0, atol=1e-5)
        assert np.abs(w - 1.0 / w.shape[1]).max() > 0.03, "degenerate (flat) softmax: the fixture would not catch a broken score path"


def _restated_variant_module(v):
    import torch

    from oracle import reference_nn as R

    kind = v["kind"]
    if kind == "projector":
        cls = {"LinearProjector": R.LinearProjector}.get(v["cls"])
        if cls is not None:
            return cls(v["vision_dim"], v["llm_dim"], pre_proj_layernorm=True)
        return getattr(R, v["cls"])(v["vision_dim"], v["llm_dim"], "gelu-mlp" if v["cls"] != "FusedMLPProjector" else "fused-gelu-mlp",
                                    pre_proj_layernorm=True)
    if kind == "attntv":
        return R.AttentivePooler(v["C"], v["llm_dim"], num_query_tokens=v["queries"], num_heads=v["heads"], output_frames=v["F"], mlp_type=v["mlp_type"])
    if kind == "conv3d":
        return R.Convolutional3DProjector(v["C"], v["llm_dim"], output_frames=v["T"], output_size=v["S"], mlp_type=v["mlp_type"])
    if kind == "concat_channel_ln":  # merv.py:219-223
        return torch.nn.Sequential(torch.nn.LayerNorm(v["E"] * v["K"]), R.LinearProjector(v["E"] * v["K"], v["K"]))
    return R.CrossAttentionAdapterLearnableQuery(embed_dim=v["embed"], llm_dim=v["K"], token_length=v["T"], averagetoken=v["averagetoken"],
                                                 num_encoder=v["E"], positional_embedding=v["pe"])


@pytest.mark.parametrize("name", _variant_names())
def test_reference_restatement_matches_reference_golden(name):
    """oracle/reference_nn.py (what the module-level tests use as the reference modules) reproduces the outputs the UNMODIFIED
    reference modules produced on the same seeded inputs and weights, every variant through its own state-dict keys."""
    import torch

    from tests.golden_util import load_variant

    v, inputs, params, gold = load_variant(name)
    m = _restated_variant_module(v).eval()
    m.load_state_dict({k: torch.from_numpy(np.ascontiguousarray(a)) for k, a in params.items()})
    xs = [torch.from_numpy(np.ascontiguousarray(x)) for x in inputs]
    with torch.no_grad():
        if v["kind"] in ("projector", "attntv", "conv3d"):
            out, w = m(xs[0]), None
        elif v["kind"] == "concat_channel_ln":  # merv.py:603-606
            out, w = m(torch.concat(xs, -1)), None
        else:
            out, w = m(xs)
    assert tuple(out.shape) == gold["out"].shape
    assert O.rel_err(out.numpy(), gold["out"]) < FP32_TOL
    if w is not None:
        assert np.abs(w.numpy() - gold["weights"]).max() < 2e-5


@pytest.mark.parametrize("name", list(C.CASES))
def test_reference_restatement_matches_reference_golden_cases(name):
    """The same for the whole fusion path of every Case (pooling resamplers + the case's mixer), against the stored samples."""
    import torch

    from oracle import reference_nn as R

    case = C.CASES[name]
    g, feats, pp, fp = regenerate(case)
    tt = lambda d: {k: torch.from_numpy(np.ascontiguousarray(a)) for k, a in d.items()}  # noqa: E731
    ys = []
    for x, p, c, t in zip(feats, pp, case.dims, case.out_frames):
        P = R.AveragePoolingProjector if case.resampler == "avg" else R.AveragePooling3DProjector
        proj = P(c, case.llm_dim, output_frames=t, output_size=case.out_size, mlp_type=case.mlp_type)
        proj.projector.load_state_dict(tt(p))
        with torch.no_grad():
            ys.append(proj(torch.from_numpy(x)))
    if case.fusion == "scalar":
        ff = R.ScalarAdapter(case.num_encoders)
    elif case.fusion == "concat_channel":
        ff = R.LinearProjector(case.num_encoders * case.llm_dim, case.llm_dim)
    else:
        ff = R.CrossAttentionAdapterLearnableQuery(embed_dim=case.embed_dim, llm_dim=case.llm_dim, token_length=case.token_length, averagetoken=True,
                                                   num_encoder=case.num_encoders)
    ff.load_state_dict(tt(fp))
    with torch.no_grad():
        if case.fusion == "concat_channel":
            out, w = ff(torch.concat(ys, -1)), None
        else:
            out, w = ff(ys)
    idx = g["sample_idx"]
    assert np.abs(out.numpy().reshape(-1)[idx] - g["out_samples"]).max() / float(g["out_abs_max"]) < FP32_TOL
    for e, y in enumerate(ys):
        ref = g["y_samples"][e]
        assert np.abs(y.numpy().reshape(-1)[idx % y.numel()] - ref).max() / max(np.abs(ref).max(), 1e-6) < FP32_TOL
    if w is not None:
        assert np.abs(w.numpy() - g["weights"]).max() < 2e-5


def test_variant_fixtures_are_sensitive_to_the_variant():
    # the positional embedding / the flattened key / the LayerNorm must move the reference's output well beyond the parity tolerance
    from tests.golden_util import load_variant

    v, inputs, params, gold = load_variant("xattn_pe")
    no_pe = {k: a for k, a in params.items() if k != "pe"}
    _, w = O.cross_attention_fusion_forward(inputs, no_pe, v["T"])
    assert np.abs(w - gold["weights"]).max() > 0.02
    v, inputs, params, gold = load_variant("pre_ln_linear")
    no_ln = {k: a for k, a in params.items() if not k.startswith("layernorm")}
    assert O.rel_err(O.projector_forward(inputs[0], no_ln, "linear"), gold["out"]) > 0.1


def test_token_concat_and_first():
    rng = np.random.default_rng(0)
    V = [rng.standard_normal((2, 3, 4)).astype(np.float32) for _ in range(3)]
    out = O.token_concat_forward(V)
    assert out.shape == (2, 9, 4) and np.array_equal(out[:, 3:6], V[1])


def test_reference_arm_port_weights_equal_the_reference_modules():
    """bench.py --impl reference builds its weights without merv_b200: the torch.nn containers of oracle/reference_model.port_state
    must consume the RNG exactly like the reference's modules (merv.py:87,152-163,214-216), and both CPU arms must agree."""
    import torch

    from oracle import reference_model as RM

    dims, llm, frames, S = [64, 48], 96, [4, 4], 2
    for mlp_type in ("linear", "gelu-mlp"):
        fwd_ref, (projs, ff) = RM.build_reference(dims, llm, frames, S, mlp_type, 16, q_scale=8.0)
        pps, fp = RM.port_state(dims, llm, mlp_type, q_scale=8.0)
        for p, sd in zip(projs, pps):
            ref_sd = p.projector.state_dict()
            assert sorted(ref_sd) == sorted(sd) and all(torch.equal(ref_sd[k], sd[k]) for k in sd)
        ref_sd = ff.state_dict()
        assert sorted(ref_sd) == sorted(fp) and all(torch.equal(ref_sd[k], fp[k]) for k in fp)
        fwd_port, _ = RM.build_port(dims, llm, frames, S, mlp_type, 16, q_scale=8.0)
        g = torch.Generator().manual_seed(3)
        feats = [torch.randn((2, 4, n, c), generator=g) + mu for n, c, mu in zip((16, 9), dims, (0.3, -0.4))]
        (o1, w1), (o2, w2) = fwd_ref(feats), fwd_port(feats)
        assert float((o1 - o2).abs().max() / o1.abs().max()) < 1e-5 and float((w1 - w2).abs().max()) < 1e-6
