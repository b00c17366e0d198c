"""Training the learnable-query adapter (``cross_attention_avg_lq``, CrossAttentionAdapterLearnableQuery) outside the configuration MERV
constructs: positional embedding (``pe`` added to each encoder's mean token, nn_utils.py:510-511), averagetoken=False (the key is the
flattened [T*K] token block, nn_utils.py:514-518 — the class default) and single-token encoders (repeated to T tokens, nn_utils.py:502).

GPU (``-m gpu``): ``ops.mix_backward_ex`` and whole ``MervFusion`` training steps against fp64 autograd through the reference modules,
bit-identity with ``ops.mix_backward`` where both apply, and bit-reproducibility.  CPU: the ABI-level argument checks, and the autograd
wiring of the modules with the kernels replaced by a torch restatement of merv_mix_backward_ex's contract.
Tolerances (max|a-b| / max|b|): fp32 2e-4, bf16 3e-2 against references at the bf16-rounded operating point.
"""
import math

import numpy as np
import pytest
import torch

from oracle import fusion_oracle as O
from oracle.cases import _uniform
from oracle.ref_loader import load_reference_nn_utils
from tests import kernel_emulation
from tests.golden_util import load_variant

DEV = "cuda:0"
TOL = {torch.float32: 2e-4, torch.bfloat16: 3e-2}
OFFSETS = (0.0, 0.5, -0.5, 0.25)


def _np(t):
    return t.detach().double().cpu().numpy()


def _round(a, dtype):
    return a if dtype == torch.float32 else torch.from_numpy(np.ascontiguousarray(a)).to(torch.bfloat16).float().numpy()


# ---- workloads ---------------------------------------------------------------------------------------------------------------------
# the three xattn variants of oracle/variants.py, plus one MERV-sized positional-embedding case and single-token encoders at bf16 tile sizes
KERNEL_CASES = {
    "xattn_flat": None,
    "xattn_pe": None,
    "xattn_pe_single": None,
    "merv_pe": dict(E=4, T=1024, K=4096, B=2, embed=3072, averagetoken=True, pe=True, single=()),
    "avg_single_wide": dict(E=4, T=256, K=1024, B=4, embed=256, averagetoken=True, pe=False, single=(1, 3)),
    "flat_single_wide": dict(E=3, T=64, K=512, B=3, embed=128, averagetoken=False, pe=False, single=(0,)),
}


def _make_case(name):
    """(settings, V list of fp32 arrays, reference state dict) of one kernel case."""
    if KERNEL_CASES[name] is None:
        v, inputs, params, _ = load_variant(name)
        return v, inputs, params
    v = KERNEL_CASES[name]
    E, T, K, B, embed, avg = v["E"], v["T"], v["K"], v["B"], v["embed"], v["averagetoken"]
    rng = np.random.default_rng(sum(map(ord, name)))
    V = [rng.standard_normal((B, 1 if e in v["single"] else T, K), dtype=np.float32) + np.float32(OFFSETS[e % 4]) for e in range(E)]
    kdim = K if avg else T * K
    xav = lambda fo, fi: math.sqrt(6.0 / (fi + fo))  # noqa: E731
    p = {
        "Q": _uniform(rng, (1, embed), xav(1, embed)) * np.float32(8.0),
        "attention.q_proj_weight": _uniform(rng, (embed, embed), xav(embed, embed)),
        "attention.k_proj_weight": _uniform(rng, (embed, kdim), xav(embed, K) / (1.0 if avg else math.sqrt(T))),
        "attention.v_proj_weight": _uniform(rng, (embed, kdim), xav(embed, K)),
        "attention.in_proj_bias": _uniform(rng, (3 * embed,), 0.05),
        "attention.out_proj.weight": _uniform(rng, (embed, embed), 1.0 / math.sqrt(embed)),
        "attention.out_proj.bias": _uniform(rng, (embed,), 0.01),
    }
    if v["pe"]:
        p["pe"] = _uniform(rng, (E, K), xav(E, K)) * np.float32(4.0)
    return v, V, p


def _loss_weights(v, seed=5):
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((v["B"], v["T"], v["K"])).astype(np.float32)
    H = rng.standard_normal((v["B"], v["E"])).astype(np.float32)
    return G, H


def _reference_adapter(v, params, device):
    ref = load_reference_nn_utils()
    m = ref.CrossAttentionAdapterLearnableQuery(embed_dim=v["embed"], llm_dim=v["K"], token_length=v["T"], averagetoken=v["averagetoken"],
                                                num_encoder=v["E"], positional_embedding=v["pe"])
    m.load_state_dict({k: torch.from_numpy(a) for k, a in params.items()})
    return m.to(device=device, dtype=torch.float64)


def _reference_kernel_grads(v, V, params, G, H, device):
    """fp64 autograd of the reference module for loss = sum(out * G) + sum(weights * H): (dV list, {param: grad})."""
    m = _reference_adapter(v, params, device)
    leaves = [torch.from_numpy(a).to(device=device, dtype=torch.float64).requires_grad_(True) for a in V]
    out, w = m(leaves)
    ((out * torch.from_numpy(G).to(device).double()).sum() + (w * torch.from_numpy(H).to(device).double()).sum()).backward()
    return [x.grad for x in leaves], {k: p.grad for k, p in m.named_parameters()}


def _kernel_inputs(v, V, params, dtype):
    """Device tensors and the forward's fp32 mixing weights (the same entry points as the module's forward)."""
    from merv_b200 import ops

    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV).to(dtype)  # noqa: E731
    Vs = [t(a) for a in V]
    Q, Wq, Wk, b = (t(params[k]) for k in ("Q", "attention.q_proj_weight", "attention.k_proj_weight", "attention.in_proj_bias"))
    pe = t(params["pe"]) if v["pe"] and v["averagetoken"] else None
    u = ops.fusion_query_vec(Q, Wq, Wk, b)
    consts = None if pe is None else ops.score_consts(pe, u)
    scores = ops.scores_from_tokens(Vs, u, v["T"], per_token_u=not v["averagetoken"], consts=consts, mean=v["averagetoken"])
    _, weights = ops.softmax_mix(Vs, v["T"], scores=scores)
    return Vs, weights, u, Q, Wq, Wk, b, pe


# ---- GPU: the kernel against the reference -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("name", list(KERNEL_CASES))
def test_mix_backward_ex_matches_reference_autograd(name, dtype):
    from merv_b200 import ops

    v, V, params = _make_case(name)
    G, H = _loss_weights(v)
    V, params, G = [_round(a, dtype) for a in V], {k: _round(a, dtype) for k, a in params.items()}, _round(G, dtype)
    want_dV, want = _reference_kernel_grads(v, V, params, G, H, DEV)
    Vs, weights, u, Q, Wq, Wk, b, pe = _kernel_inputs(v, V, params, dtype)
    dout, dw = torch.from_numpy(G).to(DEV).to(dtype), torch.from_numpy(H).to(DEV)
    dVs, dQ, dWq, dWk, dbias, dpe = ops.mix_backward_ex(Vs, dout, weights, dw, u, Q, Wq, Wk, b, per_token_u=not v["averagetoken"], pe=pe)
    tol, E = TOL[dtype], v["embed"]
    for e, (g, w_) in enumerate(zip(dVs, want_dV)):
        assert g.shape == Vs[e].shape and g.dtype == dtype
        assert O.rel_err(_np(g), _np(w_)) < tol, f"dV_{e}"
    assert O.rel_err(_np(dQ), _np(want["Q"])) < tol
    assert O.rel_err(_np(dWq), _np(want["attention.q_proj_weight"])) < tol
    assert dWk.shape == Wk.shape and O.rel_err(_np(dWk), _np(want["attention.k_proj_weight"])) < tol
    assert O.rel_err(_np(dbias)[:E], _np(want["attention.in_proj_bias"])[:E]) < tol
    assert not dbias[E:].any()  # b_k cancels in the softmax, b_v is dead
    if pe is not None:
        assert dpe.shape == pe.shape and O.rel_err(_np(dpe), _np(want["pe"])) < tol
    else:
        assert dpe is None


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shape", [(3, 4, 256, 1024, 256), (2, 3, 64, 1000, 96), (16, 4, 1024, 4096, 3072)], ids=["wide", "ragged_k", "merv_b16"])
def test_mix_backward_ex_is_mix_backward_on_the_shipped_configuration(shape, dtype):
    """All encoders at T tokens, averagetoken=True, no positional embedding: the new entry point and the old one agree bit for bit."""
    from merv_b200 import ops

    B, E, T, K, embed = shape
    g = torch.Generator(device=DEV).manual_seed(11)
    Vs = [(torch.randn(B, T, K, generator=g, device=DEV) + OFFSETS[e]).to(dtype) for e in range(E)]
    Q, Wq, Wk, b = ((torch.randn(*s, generator=g, device=DEV) * sc).to(dtype)
                    for s, sc in (((1, embed), 4.0), ((embed, embed), embed ** -0.5), ((embed, K), K ** -0.5), ((3 * embed,), 0.05)))
    u = ops.fusion_query_vec(Q, Wq, Wk, b)
    _, weights = ops.softmax_mix(Vs, T, scores=ops.scores_from_tokens(Vs, u, T))
    dout = torch.randn(B, T, K, generator=g, device=DEV).to(dtype)
    dw = torch.randn(B, E, generator=g, device=DEV)
    old = ops.mix_backward(Vs, dout, weights, dw, u, Q, Wq, Wk, b)
    new = ops.mix_backward_ex(Vs, dout, weights, dw, u, Q, Wq, Wk, b)
    assert new[5] is None
    for e in range(E):
        assert torch.equal(old[0][e], new[0][e]), f"dV_{e}"
    for i, what in enumerate(("dQ", "dWq", "dWk", "dbias"), start=1):
        assert torch.equal(old[i], new[i]), what


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("name", ["xattn_flat", "xattn_pe_single", "avg_single_wide", "flat_single_wide"])
def test_mix_backward_ex_is_bit_reproducible(name, dtype):
    from merv_b200 import ops

    v, V, params = _make_case(name)
    G, H = _loss_weights(v)
    Vs, weights, u, Q, Wq, Wk, b, pe = _kernel_inputs(v, V, params, dtype)
    dout, dw = torch.from_numpy(G).to(DEV).to(dtype), torch.from_numpy(H).to(DEV)
    run = lambda: ops.mix_backward_ex(Vs, dout, weights, dw, u, Q, Wq, Wk, b, per_token_u=not v["averagetoken"], pe=pe)  # noqa: E731
    first, second = run(), run()
    for a, c in zip(first[0], second[0]):
        assert torch.equal(a, c)
    for a, c in zip(first[1:], second[1:]):
        assert (a is None and c is None) or torch.equal(a, c)


# ---- module level: MervFusion training steps -------------------------------------------------------------------------------------------
# 3davg + linear projectors (channels 32 / 48 / 64, 4 frames of 4 x 4 patches -> 2 x 2 x 2 = 8 tokens; an encoder in `single` pools to
# 1 x 1 x 1: a single token) in front of the adapter in each configuration
MODULE_CONFIGS = {
    "pe": dict(averagetoken=True, pe=True, single=()),
    "pe_single": dict(averagetoken=True, pe=True, single=(1,)),
    "avg_single": dict(averagetoken=True, pe=False, single=(2,)),
    "flat": dict(averagetoken=False, pe=False, single=()),
    "flat_single_pe": dict(averagetoken=False, pe=True, single=(0,)),  # pe exists but the reference never reads it
}
_DIMS, _K, _EMBED, _B, _F, _N = (32, 48, 64), 64, 48, 2, 4, 16


def _module_setup(cfg, dtype):
    """(reference projectors, reference adapter, features, G, H) with seeded parameters, rounded to the bf16 operating point if needed."""
    ref = load_reference_nn_utils()
    c = MODULE_CONFIGS[cfg]
    torch.manual_seed(7)
    projs = [ref.AveragePooling3DProjector(C, _K, 1 if e in c["single"] else 2, 1 if e in c["single"] else 2, mlp_type="linear")
             for e, C in enumerate(_DIMS)]
    ff = ref.CrossAttentionAdapterLearnableQuery(embed_dim=_EMBED, llm_dim=_K, token_length=8, averagetoken=c["averagetoken"], num_encoder=len(_DIMS),
                                                 positional_embedding=c["pe"])
    with torch.no_grad():
        ff.Q.mul_(8.0)  # a mixing softmax far from uniform
        if c["pe"]:
            ff.pe.mul_(4.0)
        for m in projs + [ff]:
            for p in m.parameters():
                p.copy_(torch.from_numpy(_round(p.detach().numpy(), dtype)))
    g = torch.Generator().manual_seed(3)
    xs = [torch.from_numpy(_round((torch.randn(_B, _F, _N, C, generator=g) + OFFSETS[e]).numpy(), dtype)) for e, C in enumerate(_DIMS)]
    G = torch.from_numpy(_round(torch.randn(_B, 8, _K, generator=g).numpy(), dtype))
    H = torch.randn(_B, len(_DIMS), generator=g)
    return projs, ff, xs, G, H


def _check_module_training(cfg, dtype, device):
    import merv_b200 as M

    c = MODULE_CONFIGS[cfg]
    rprojs, rff, xs, G, H = _module_setup(cfg, dtype)
    projs = [M.AveragePooling3DProjector(p.projector.projector.in_features, _K, p.output_frames, p.output_size, "linear") for p in rprojs]
    for p, r in zip(projs, rprojs):
        p.load_state_dict(r.state_dict())
    ff = M.CrossAttentionAdapterLearnableQuery(_EMBED, _K, 8, averagetoken=c["averagetoken"], num_encoder=len(_DIMS), positional_embedding=c["pe"])
    ff.load_state_dict(rff.state_dict())
    m = M.MervFusion(projs, ff).to(device=device, dtype=dtype).train()

    # reference: fp64 autograd through the reference modules
    rprojs = [p.double() for p in rprojs]
    rff = rff.double()
    want_out, want_w = rff([p(x.double()) for p, x in zip(rprojs, xs)])
    ((want_out * G.double()).sum() + (want_w * H.double()).sum()).backward()

    out, w = m([x.to(device=device, dtype=dtype) for x in xs])
    assert type(out.grad_fn).__name__.startswith("_MixFn")  # linked projectors hand over DeferredProjections, materialised for autograd
    tol = TOL[dtype]
    assert O.rel_err(_np(out), _np(want_out)) < tol and O.rel_err(_np(w), _np(want_w)) < tol
    ((out.float() * G.to(device)).sum() + (w.float() * H.to(device)).sum()).backward()
    for i, (p, r) in enumerate(zip(m.projectors, rprojs)):
        got, ref = dict(p.named_parameters()), dict(r.named_parameters())
        assert sorted(got) == sorted(ref)
        for k in ref:
            assert got[k].grad is not None and O.rel_err(_np(got[k].grad), _np(ref[k].grad)) < tol, f"projector {i} {k}"
    att, ratt, E = m.feature_fusion.attention, rff.attention, _EMBED
    assert O.rel_err(_np(m.feature_fusion.Q.grad), _np(rff.Q.grad)) < tol
    assert O.rel_err(_np(att.q_proj_weight.grad), _np(ratt.q_proj_weight.grad)) < tol
    assert O.rel_err(_np(att.k_proj_weight.grad), _np(ratt.k_proj_weight.grad)) < tol
    assert O.rel_err(_np(att.in_proj_bias.grad)[:E], _np(ratt.in_proj_bias.grad)[:E]) < tol
    assert not att.in_proj_bias.grad[E:].any()  # b_k and b_v: exactly zero
    assert att.v_proj_weight.grad is None and att.out_proj.weight.grad is None and att.out_proj.bias.grad is None
    assert ratt.v_proj_weight.grad is None
    if c["pe"] and c["averagetoken"]:
        assert O.rel_err(_np(m.feature_fusion.pe.grad), _np(rff.pe.grad)) < tol
    elif c["pe"]:
        assert m.feature_fusion.pe.grad is None and rff.pe.grad is None


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("cfg", list(MODULE_CONFIGS))
def test_merv_fusion_training_matches_reference_autograd(cfg, dtype):
    _check_module_training(cfg, dtype, DEV)


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------------
def _mix_backward_ex_standin(Vs, dout, weights, dweights, u, Q, Wq, Wk, in_proj_bias, per_token_u=False, pe=None):
    """merv_mix_backward_ex's contract (include/merv_fusion.h) restated with torch autograd: the stand-in the CPU wiring test routes to."""
    B, T, K = dout.shape
    E, embed, dt = len(Vs), Wk.shape[0], Vs[0].dtype
    leaves = [t.float().clone().requires_grad_(True) for t in (*Vs, Q, Wq, Wk, in_proj_bias, *([] if pe is None else [pe]))]
    with torch.enable_grad():
        Vf, (Qf, Wqf, Wkf, bf) = leaves[:E], leaves[E:E + 4]
        uu = ((Qf.reshape(1, embed) @ Wqf.T + bf[:embed]) @ Wkf)[0] / math.sqrt(embed)
        full = [v.expand(-1, T, -1) for v in Vf]
        if per_token_u:
            scores = torch.stack([v.reshape(B, T * K) @ uu for v in full], 1)
        else:
            scores = torch.stack([(v.mean(1) + (leaves[-1][e] if pe is not None else 0.0)) @ uu for e, v in enumerate(full)], 1)
        w = torch.softmax(scores, -1)
        out = sum(w[:, e, None, None] * v for e, v in enumerate(full))
        loss = (out * dout.float()).sum() + (0.0 if dweights is None else (w * dweights).sum())
    g = [t.to(dt) for t in torch.autograd.grad(loss, leaves)]
    return g[:E], g[E].reshape(1, embed), g[E + 1], g[E + 2], g[E + 3], (g[E + 4] if pe is not None else None)


@pytest.mark.parametrize("cfg", list(MODULE_CONFIGS))
def test_training_wiring_matches_reference_on_cpu(cfg, monkeypatch):
    """The module code unchanged, the kernels emulated: _MixFn is reached through the deferred projections, gets ``pe`` exactly when the
    reference reads it, and hands the right tensors to mix_backward_ex."""
    from merv_b200 import ops

    kernel_emulation.emulate(monkeypatch)
    calls = []

    def standin(*a, **kw):
        calls.append(kw)
        return _mix_backward_ex_standin(*a, **kw)

    monkeypatch.setattr(ops, "mix_backward_ex", standin)
    _check_module_training(cfg, torch.float32, "cpu")
    c = MODULE_CONFIGS[cfg]
    assert len(calls) == 1 and calls[0]["per_token_u"] == (not c["averagetoken"])
    assert (calls[0]["pe"] is not None) == (c["pe"] and c["averagetoken"])


@pytest.mark.parametrize("name", ["xattn_flat", "xattn_pe", "xattn_pe_single"])
def test_variant_adapter_gradients_on_cpu(name, monkeypatch):
    """The xattn variants with the token tensors themselves requiring grad (no projectors in front)."""
    import merv_b200 as M
    from merv_b200 import ops

    kernel_emulation.emulate(monkeypatch)
    monkeypatch.setattr(ops, "mix_backward_ex", _mix_backward_ex_standin)
    v, V, params = _make_case(name)
    G, H = _loss_weights(v)
    want_dV, want = _reference_kernel_grads(v, V, params, G, H, "cpu")
    ff = M.CrossAttentionAdapterLearnableQuery(embed_dim=v["embed"], llm_dim=v["K"], token_length=v["T"], averagetoken=v["averagetoken"],
                                               num_encoder=v["E"], positional_embedding=v["pe"])
    ff.load_state_dict({k: torch.from_numpy(a) for k, a in params.items()})
    leaves = [torch.from_numpy(a).requires_grad_(True) for a in V]
    out, w = ff(leaves)
    assert type(out.grad_fn).__name__.startswith("_MixFn")
    ((out * torch.from_numpy(G)).sum() + (w * torch.from_numpy(H)).sum()).backward()
    for x, r in zip(leaves, want_dV):
        assert x.grad.shape == x.shape and O.rel_err(_np(x.grad), _np(r)) < 1e-4
    for k, p in ff.named_parameters():
        if want[k] is None:
            assert p.grad is None or not p.grad.any(), k
        elif k == "attention.in_proj_bias":
            assert O.rel_err(_np(p.grad)[:v["embed"]], _np(want[k])[:v["embed"]]) < 1e-4 and not p.grad[v["embed"]:].any()
        else:
            assert O.rel_err(_np(p.grad), _np(want[k])) < 1e-4, k


def test_mix_backward_ex_workspace_and_argument_checks():
    """Checks that run before any device is touched: the workspace sizes and the rejected argument combinations."""
    import ctypes

    from merv_b200 import _lib

    lib = _lib.load()
    B, E, T, K, embed = 4, 3, 16, 64, 32
    old = lib.merv_mix_backward_workspace(B, E, T, K, embed)
    assert lib.merv_mix_backward_ex_workspace(B, E, T, K, embed, 0) == old + B * K  # + the single-token column sums
    assert lib.merv_mix_backward_ex_workspace(B, E, T, K, embed, K) == old + (T - 1) * K + B * K  # du is [T*K]
    fake = ctypes.c_void_p(256)  # never dereferenced: every check below fails before a device is touched
    ptrs = _lib.ptr_array([256] * E)
    tokens = _lib.i32_array([T] * E)

    def call(stride, pe, dpe, ldpe=K):
        return lib.merv_mix_backward_ex(ptrs, tokens, fake, fake, None, fake, stride, pe, ldpe, fake, fake, fake, fake, ptrs, fake, fake, fake, fake,
                                        dpe, fake, 1 << 20, B, E, T, K, embed, _lib.MERV_BF16, None)

    assert call(K, fake, fake) == -6 and b"pe" in lib.merv_last_error()  # averagetoken=False never reads pe
    assert call(0, fake, None) == -6 and b"dpe" in lib.merv_last_error()
    assert call(0, fake, fake, ldpe=K - 8) == -1
    assert call(K // 2, None, None) == -1 and b"u_token_stride" in lib.merv_last_error()
