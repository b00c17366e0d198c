"""The kernels of the fused backward, called directly and compared element by element with fp64 references.

The fused training step (``_FusedLinearFn`` in front of the learnable-query mixer, ``_FusedScalarLinearFn`` in front of the scalar mixer)
never writes the per-encoder projections Y_e or their gradients.  All of its gradients come from ``merv_wgrad_video`` (or, when the token
count is not a multiple of 64, the two MN-major ``merv_gemm_ex`` GEMMs with ``merv_pair_dot_scale``), ``merv_video_colsum`` and
``merv_fused_backward`` / ``merv_scalar_fused_backward``.  Each is tested here on its own at the shapes where its branches and tiling
change, and the whole chain is composed by hand from the same calls and checked against fp64 closed forms.

Every reference is fp64, computed from the inputs the kernel actually received (bf16 operands are already rounded, fp32 intermediates are
the kernel's own), and every check is per element through ``check_bound`` of the forward file, which names the worst element in kernel
terms (row block, column tile, epilogue group and split range of a weight gradient; video; output, encoder, row and column).

Error model, with u = 2^-24 and ``mag`` the fp64 expression with every operand and every intermediate sum replaced by its absolute value:
``bound = r |ref| + 4 u depth mag``, r = 2^-8 for a bf16 output (its rounding) and u for an fp32 one, ``depth`` the longest chain of
fp32 operations behind the element:

* ``dW`` of ``merv_wgrad_video``: T tensor-core products per video, the ``videos`` scaled adds of the epilogue's running sum, and the
  ``split`` partial tiles of the fold: depth T + videos + split + 2.
* its per-video dot (the sum of the video's 32 chunks): the accumulator (T), the epilogue's 64-column fma chain and 32-lane tree
  (64 + 5), and ceil(parts / 32) partials per chunk in the fold: depth T + 69 + ceil(parts / 32) + 2.
* ``merv_fused_backward``: dw_e = sum of the pair-dot partials + b_e . gsum is a ceil(K / 32) fma chain per lane, a 5-level warp tree and
  the dweights_out add; ds = w (.) (dw - <w, dw>) adds E + 8 levels.  ``mag(ds)`` is taken through the softmax backward from ``mag(dw)``:
  |w| (mag(dw) + <|w|, mag(dw)>).  g_e, db_e, the rank-1 term u (x) g_e, du, q, dq, dWk, dWq and dQ propagate ``mag`` the same way, each
  adding the length of its own reduction (B videos, ceil(C_e / 32) + 5 per encoder row, ceil(K / 32) + 5, embed / 64 + 16 for the
  two-stage dQ) plus a few roundings (the fp32 1/sqrt(embed)).  The in_proj_bias gradient past ``embed`` is exactly 0.
* ``dW_e`` of a whole step is rounded to bf16 twice, by the GEMM and again by the in-place rank-1 update, so its bound carries both
  roundings: 2^-8 |GEMM part| + 2^-8 |ref|.  In the two-GEMM form Z_e = dOut W_e and w_e (.) P_e are stored in bf16 before they are
  reduced, which adds 2^-8 of the magnitude of everything computed from them.
* ``merv_scalar_fused_backward``: gs = sum over B videos, db_e = w_e gs, g_e = partials + b_e . gs + dweights_out through a 256-thread
  block sum (two 5-level warp trees) and a final CTA that adds its share serially, then a warp tree and its 8 warps in order (13 levels);
  dscalar = w (.) (g - <w, g>) adds one more warp tree and two operations.
* ``merv_video_colsum``: ceil(T / 32) adds per thread, the 32 row groups in order and the scale.  ``merv_colsum``: per 256-row block
  8 + 32 (vector path) or 256 (scalar path), then the ceil(M / 256) block sums.  ``merv_pair_dot``: per chunk, the thread's fma chain of
  at most ceil(per / 256) vectors and the 256-thread block sum (10 levels).  ``y_scaled`` and ``merv_transpose_rowscale`` are one fp32
  multiply and one rounding: bit-identical to torch.

The modules' own backward (``MervFusion(fused_training=True)``) is asserted bit-identical to the hand composition of the same calls, so the
glue in ``merv_b200/nn_utils.py`` is pinned as well as the kernels.

The CPU tests below show that the harness catches the mistakes it is meant to catch (the rounded fp64 reference with one mutation at a
time), and that the closed forms equal fp64 autograd through the reference modules.
"""
import ctypes
import math

import pytest
import torch

from tests.test_fused_forward_kernels import BF16_REL, TINY, U, GemmLayout, VideoLayout, check_bound, gemm_bound  # noqa: F401

DEV = "cuda:0"
CHUNKS = 32  # merv_pair_dot_chunks()
EPI_COLS, WARP_LEVELS = 64, 5


# ---- layouts -----------------------------------------------------------------------------------------------------------------------
class WgradLayout:
    """Names an element of dW [N_out, C] of merv_wgrad_video: its row and 128-row block (256 for a CTA pair), its column, 256-column tile
    and 64-column epilogue group, and the contiguous video ranges of the split (every range contributes to every element)."""

    def __init__(self, videos, split, ctas):
        self.rows = 128 * ctas
        self.ranges = [(q * videos) // split for q in range(split + 1)]

    def describe(self, idx):
        n, c = idx
        rng = ", ".join(f"[{a}, {b})" for a, b in zip(self.ranges[:-1], self.ranges[1:]))
        return (f"dW row {n} ({self.rows}-row block {n // self.rows}), column {c} (256-column tile {c // 256}, 64-column epilogue group "
                f"{(c % 256) // EPI_COLS}), split ranges of videos {rng}")


class DotLayout:
    """Per-video dots [videos] (or per-chunk [videos, chunks])."""

    def describe(self, idx):
        return f"dot of video {idx[0]}" + (f", chunk {idx[1]}" if len(idx) > 1 else "")


class OutLayout:
    """An output of merv_fused_backward / merv_scalar_fused_backward: its name, encoder, and the index named per dimension."""

    def __init__(self, name, dims, encoder=None):
        self.name, self.dims, self.encoder = name, dims, encoder

    def describe(self, idx):
        enc = "" if self.encoder is None else f" of encoder {self.encoder}"
        return f"{self.name}{enc}, " + ", ".join(f"{d} {i}" for d, i in zip(self.dims, idx))


def _rnd(dtype):
    return BF16_REL if dtype == torch.bfloat16 else U


def _bound(ref, mag, depth, dtype, eps=0.0):
    return _rnd(dtype) * ref.abs() + (eps + 4 * U * depth) * mag


# ---- fp64 references -------------------------------------------------------------------------------------------------------------
def wgrad_reference(dy, x, scale, w):
    """dy [V, T, N], x [V, T, C], scale [V], w [N, C] -> (dW, mag(dW), dot [V], mag(dot)) of dW = sum_b s_b dy_b^T x_b, dot_b = <w, dy_b^T x_b>."""
    V, T, N = dy.shape
    d, xx, s = dy.double(), x.double(), scale.double().reshape(V, 1, 1)
    ref = (d * s).reshape(V * T, N).T @ xx.reshape(V * T, -1)
    mag = (d.abs() * s.abs()).reshape(V * T, N).T @ xx.abs().reshape(V * T, -1)
    w64 = w.double()
    dot = (d * (xx @ w64.T)).sum((1, 2))
    mdot = (d.abs() * (xx.abs() @ w64.abs().T)).sum((1, 2))
    return ref, mag, dot, mdot


def wgrad_bounds(ref, mag, dot, mdot, T, videos, split, parts):
    return (_bound(ref, mag, T + videos + split + 2, torch.bfloat16),
            4 * U * (T + EPI_COLS + WARP_LEVELS + math.ceil(parts / CHUNKS) + 2) * mdot)


def fused_bwd_reference(weights, dwo, u, gsum, parts, pbar, Ws, biases, Q, Wq, Wk, ipb, dW_in):
    """fp64 closed forms of merv_fused_backward (include/merv_fusion.h above merv_fused_bwd_desc).

    Stage inputs come as (value, mag) pairs so that the same code serves the kernel's own inputs (mag = |value|) and a whole step (mag
    carried from the tokens): gsum [B, K], parts[e] [B, n] (summed over n), pbar[e] [B, C_e], dW_in[e] [K, C_e] or None.
    Returns {name: (ref, mag, depth)} with names ds, dW{e}, db{e}, dQ, dWq, dWk, dbias."""
    d = lambda t: None if t is None else t.double()  # noqa: E731
    w = d(weights)
    aw = w.abs()
    B, E = w.shape
    K, embed = u.numel(), Wk.shape[0]
    u64 = d(u)
    gs, mgs = gsum
    dw, mdw = [], []
    for e in range(E):
        pv, pm = parts[e]
        v, m = pv.sum(1), pm.sum(1)
        if biases[e] is not None:
            b = d(biases[e])
            v, m = v + gs @ b, m + mgs @ b.abs()
        dw.append(v)
        mdw.append(m)
    dw, mdw = torch.stack(dw, 1), torch.stack(mdw, 1)
    if dwo is not None:
        dw, mdw = dw + d(dwo), mdw + d(dwo).abs()
    ds = w * (dw - (w * dw).sum(1, keepdim=True))
    mds = aw * (mdw + (aw * mdw).sum(1, keepdim=True))
    n_ds = math.ceil(K / 32) + WARP_LEVELS + 2 + E + 8
    out = {"ds": (ds, mds, n_ds)}
    sig, msig = ds.sum(0), mds.sum(0)
    n_g = n_ds + B + 1
    du = torch.zeros(K, dtype=torch.float64, device=w.device)
    mdu = torch.zeros_like(du)
    cmax = 0
    for e in range(E):
        pb, mpb = pbar[e]
        g, mg = ds[:, e] @ pb, mds[:, e] @ mpb
        r1, mr1 = torch.outer(u64, g), torch.outer(u64.abs(), mg)
        if dW_in[e] is not None:
            wv, wm = dW_in[e]
            out[f"dW{e}"] = (wv + r1, wm + mr1, n_g + 2)
        gsum_w = w[:, e] @ gs
        out[f"db{e}"] = (gsum_w + u64 * sig[e], aw[:, e] @ mgs + u64.abs() * msig[e], n_ds + B + 2)
        We = d(Ws[e])
        du, mdu = du + We @ g, mdu + We.abs() @ mg
        if biases[e] is not None:
            b = d(biases[e])
            du, mdu = du + sig[e] * b, mdu + msig[e] * b.abs()
        cmax = max(cmax, We.shape[1])
    n_du = n_g + math.ceil(cmax / 32) + WARP_LEVELS + B + E + 2
    Q64, Wq64, Wk64 = d(Q).reshape(-1), d(Wq), d(Wk)
    q, mq = Wq64 @ Q64, Wq64.abs() @ Q64.abs()
    if ipb is not None:
        bq = d(ipb)[:embed]
        q, mq = q + bq, mq + bq.abs()
    n_q = math.ceil(embed / 32) + WARP_LEVELS + 2
    rs = 1.0 / math.sqrt(embed)
    dq, mdq = rs * (Wk64 @ du), rs * (Wk64.abs() @ mdu)
    n_dq = n_du + math.ceil(K / 32) + WARP_LEVELS + 4
    out["dWk"] = (rs * torch.outer(q, du), rs * torch.outer(mq, mdu), n_du + n_q + 4)
    out["dWq"] = (torch.outer(dq, Q64), torch.outer(mdq, Q64.abs()), n_dq + 1)
    out["dQ"] = ((Wq64.T @ dq)[None], (Wq64.abs().T @ mdq)[None], n_dq + math.ceil(embed / 64) + 16)
    z = torch.zeros(2 * embed, dtype=torch.float64, device=w.device)
    out["dbias"] = (torch.cat([dq, z]), torch.cat([mdq, z]), n_dq)
    out["du"] = (du, mdu, n_du)
    return out


def scalar_fused_reference(weights, dwo, gsum, parts, biases):
    """fp64 closed forms of merv_scalar_fused_backward: {name: (ref, mag, depth)} for dscalar and db{e}; gsum and parts[e] are tensors
    (mag = |value|) or (value, mag) pairs."""
    w = weights.double()
    E = w.numel()
    gv, gm = gsum if isinstance(gsum, tuple) else (gsum.double(), gsum.double().abs())
    B, K = gv.shape
    gs, mgs = gv.sum(0), gm.sum(0)
    g, mg = [], []
    for e in range(E):
        pv, pm = parts[e] if isinstance(parts[e], tuple) else (parts[e].double(), parts[e].double().abs())
        v, m = pv.sum(), pm.sum()
        if biases[e] is not None:
            b = biases[e].double()
            v, m = v + gs @ b, m + mgs @ b.abs()
        g.append(v)
        mg.append(m)
    g, mg = torch.stack(g), torch.stack(mg)
    if dwo is not None:
        g, mg = g + dwo.double(), mg + dwo.double().abs()
    nb = -(-K // 256)
    # gs: B serial adds; b_e . gs: one product, then a 256-thread block sum (two 5-level warp trees) per CTA; stage 2: each thread adds
    # ceil(B * 32 / 256) partials and ceil(nb / 256) CTA sums, then a 5-level warp tree and the 8 warps' sums in order (13), then
    # dweights_out; dscalar = w (.) (g - <w, g>): one more 5-level tree for <w, g>, the subtraction and the product
    n_g = B + 1 + 10 + math.ceil(B * CHUNKS / 256) + math.ceil(nb / 256) + 13 + 1
    out = {"dscalar": (w * (g - (w * g).sum()), w.abs() * (mg + (w.abs() * mg).sum()), n_g + 5 + 2)}
    for e in range(E):
        out[f"db{e}"] = (w[e] * gs, w[e].abs() * mgs, B + 1)
    return out


def closed_form_step(P, Ws, biases, G, weights, dwo, u, Q, Wq, Wk, ipb):
    """fp64 gradients of one fused learnable-query step from its pooled tokens P_e [B, T, C_e], the gradient G [B, T, K] of the fused
    tokens, the forward's mixing weights [B, E] and u: the stage inputs are formed exactly, with their magnitudes, and handed to
    fused_bwd_reference.  Also returns the GEMM part dOut^T (w_e (.) P_e) of every dW_e, for the double rounding of a whole step."""
    B, T, K = G.shape
    G64 = G.double()
    gs, mgs = G64.sum(1), G64.abs().sum(1)
    parts, pbars, dW_in, gemm = [], [], [], []
    for e, p in enumerate(P):
        p64, W64 = p.double(), Ws[e].double()
        Z, mZ = G64 @ W64, G64.abs() @ W64.abs()
        parts.append(((Z * p64).sum((1, 2))[:, None], (mZ * p64.abs()).sum((1, 2))[:, None]))
        pbars.append((p64.mean(1), p64.abs().mean(1)))
        wv = weights[:, e].double()[:, None, None]
        dWv = G64.reshape(B * T, K).T @ (wv * p64).reshape(B * T, -1)
        dWm = G64.abs().reshape(B * T, K).T @ (wv.abs() * p64.abs()).reshape(B * T, -1)
        dW_in.append((dWv, dWm))
        gemm.append(dWv)
    out = fused_bwd_reference(weights, dwo, u, (gs, mgs), parts, pbars, Ws, biases, Q, Wq, Wk, ipb, dW_in)
    return out, gemm


# ---- the harness catches what it must (CPU) --------------------------------------------------------------------------------------------
SELF_V, SELF_T, SELF_N, SELF_C, SELF_SPLIT = 10, 128, 40, 24, 3


def _video_scales(V):
    """Neighbouring videos differ by at least 0.1; video V // 2 has scale 0, video 1 a negative one."""
    s = 0.3 + 0.15 * torch.remainder(3 * torch.arange(V, dtype=torch.float64), 7)
    if V >= 3:
        s[V // 2] = 0.0
    if V >= 2:
        s[1] = -s[1]
    return s.float()


def _wgrad_case(V, T, N, C, seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    dy = (torch.randn(V, T, N, generator=g) + 0.2).to(torch.bfloat16)
    x = (torch.rand(V, T, C, generator=g) + 0.1).to(torch.bfloat16)
    w = ((torch.rand(N, C, generator=g) - 0.3) / math.sqrt(C)).to(torch.bfloat16)
    return dy.to(device), x.to(device), _video_scales(V).to(device), w.to(device)


@pytest.fixture(scope="module")
def wgrad_self_case():
    dy, x, s, w = _wgrad_case(SELF_V, SELF_T, SELF_N, SELF_C, seed=5)
    ref, mag, dot, mdot = wgrad_reference(dy, x, s, w)
    bdw, bdot = wgrad_bounds(ref, mag, dot, mdot, SELF_T, SELF_V, SELF_SPLIT, parts=16)
    return dy, x, s, w, ref, bdw, dot, bdot


def test_wgrad_bound_passes_the_rounded_reference(wgrad_self_case):
    *_, ref, bdw, dot, bdot = wgrad_self_case
    check_bound(ref.to(torch.bfloat16), ref, bdw, WgradLayout(SELF_V, SELF_SPLIT, 1))
    check_bound(dot.float(), dot, bdot, DotLayout())


@pytest.mark.parametrize("kind", ["scales_swapped_at_split_boundary", "dropped_last_k_block", "dots_swapped"])
def test_wgrad_bound_fails_on_each_mutation(wgrad_self_case, kind):
    """A per-video dot is caught with its video named.  An element of dW sums over every video, so no single video can be named there:
    the message must name the worst element itself (row, row block, column, column tile, epilogue group) with the split ranges."""
    dy, x, s, w, ref, bdw, dot, bdot = wgrad_self_case
    layout = WgradLayout(SELF_V, SELF_SPLIT, 1)
    dot_where, check_dw = None, True
    if kind == "scales_swapped_at_split_boundary":  # videos 2 and 3 sit on either side of the first boundary of 3 ranges over 10 videos
        assert layout.ranges[1] == 3 and abs(float(s[2] - s[3])) >= 0.1
        s2 = s.clone()
        s2[[2, 3]] = s2[[3, 2]]
        got_ref, _, got_dot, _ = wgrad_reference(dy, x, s2, w)
    elif kind == "dropped_last_k_block":  # video 4 loses its last 64 tokens
        dy2 = dy.clone()
        dy2[4, -64:] = 0
        got_ref, _, got_dot, _ = wgrad_reference(dy2, x, s, w)
        dot_where = ("dot of video 4",)
    else:
        got_ref, got_dot = ref, dot.clone()
        got_dot[[6, 7]] = got_dot[[7, 6]]
        dot_where, check_dw = ("dot of video 6", "dot of video 7"), False
    got = got_ref.to(torch.bfloat16)
    if not check_dw:
        check_bound(got, ref, bdw, layout)
    else:
        with pytest.raises(AssertionError, match="out of bound") as e:
            check_bound(got, ref, bdw, layout)
        ratio = (got.double() - ref).abs() / bdw
        n, c = (int(i) for i in torch.unravel_index(torch.argmax(ratio), ratio.shape))
        assert f"worst at {layout.describe((n, c))}:" in str(e.value), str(e.value)
        assert "split ranges of videos [0, 3), [3, 6), [6, 10)" in str(e.value)
    if dot_where is None:
        check_bound(got_dot.float(), dot, bdot, DotLayout())
    else:
        with pytest.raises(AssertionError, match="out of bound") as e:
            check_bound(got_dot.float(), dot, bdot, DotLayout())
        assert any(wh in str(e.value) for wh in dot_where), str(e.value)


def _step_case(B, T, Cs, K, embed, seed, device="cpu", dtype=torch.bfloat16):
    """Inputs of one learnable-query step: pooled tokens with positive means, distinct weight rows, dweights_out large enough that ds
    (and with it the rank-1 term, db's u-term and du) is well above the rounding of the larger terms."""
    g = torch.Generator().manual_seed(seed)
    E = len(Cs)
    P = [(torch.rand(B, T, c, generator=g) + 0.2).to(dtype) for c in Cs]
    Ws = [((torch.rand(K, c, generator=g) - 0.3) / math.sqrt(c)).to(dtype) for c in Cs]
    biases = [None if e == 1 else (torch.randn(K, generator=g) * 0.5).to(dtype) for e in range(E)]
    G = (torch.randn(B, T, K, generator=g) * 0.5 + 0.1).to(dtype)
    scores = torch.randn(B, E, generator=g) + 0.5 * torch.arange(B)[:, None] % 3
    weights = torch.softmax(scores, -1).float()
    dwo = torch.randn(B, E, generator=g) * 4
    Q = torch.randn(1, embed, generator=g).to(dtype)
    Wq = (torch.randn(embed, embed, generator=g) / math.sqrt(embed)).to(dtype)
    Wk = (torch.randn(embed, K, generator=g) / math.sqrt(embed)).to(dtype)
    ipb = (torch.randn(3 * embed, generator=g) * 0.3).to(dtype)
    q = Wq.double() @ Q.double()[0] + ipb.double()[:embed]
    u = ((Wk.double().T @ q) / math.sqrt(embed)).float()
    mv = lambda t: None if t is None else t.to(device)  # noqa: E731
    return ([mv(p) for p in P], [mv(w) for w in Ws], [mv(b) for b in biases], mv(G), mv(weights), mv(dwo), mv(u), mv(Q), mv(Wq), mv(Wk),
            mv(ipb))


SELF_STEP = dict(B=6, T=8, Cs=(24, 16, 40), K=48, embed=16)


@pytest.fixture(scope="module")
def step_self_case():
    args = _step_case(**SELF_STEP, seed=3)
    out, _ = closed_form_step(*args)
    return args, out


def _step_layouts(name):
    if name == "ds":
        return OutLayout("ds", ("video", "encoder"))
    if name.startswith("dW") and name[2:].isdigit():
        return OutLayout("dW", ("row", "column"), int(name[2:]))
    if name.startswith("db") and name[2:].isdigit():
        return OutLayout("db", ("row",), int(name[2:]))
    return OutLayout(name, ("row", "column") if name in ("dWq", "dWk", "dQ") else ("element",))


def _check_step(got, out, dtype=torch.bfloat16):
    for name, (ref, mag, depth) in out.items():
        if name == "du":
            continue
        check_bound(got[name], ref, _bound(ref, mag, depth, dtype), _step_layouts(name))


def test_step_bound_passes_the_rounded_reference(step_self_case):
    _, out = step_self_case
    _check_step({k: v[0].to(torch.bfloat16) if k != "ds" else v[0].float() for k, v in out.items()}, out)


def _mutated_step(args, out, kind):
    P, Ws, biases, G, weights, dwo, u, Q, Wq, Wk, ipb = args
    got = {k: v[0].clone() for k, v in out.items()}
    B = weights.shape[0]
    if kind == "rank1_left_out":  # encoder 2's dW without u (x) g_2
        ds = out["ds"][0]
        g2 = ds[:, 2] @ P[2].double().mean(1)
        got["dW2"] = got["dW2"] - torch.outer(u.double(), g2)
    elif kind == "ds_swapped":  # videos 3 and 4
        assert (out["ds"][0][3] - out["ds"][0][4]).abs().max() > 0.1
        got["ds"] = got["ds"][[*range(3), 4, 3, *range(5, B)]]
    elif kind == "db_without_u_term":  # encoder 0
        got["db0"] = got["db0"] - u.double() * out["ds"][0][:, 0].sum()
    elif kind == "dQ_not_transposed":
        dq = out["dbias"][0][:Q.shape[1]]
        got["dQ"] = (Wq.double() @ dq)[None]
    else:
        raise ValueError(kind)
    return {k: v.to(torch.bfloat16) if k != "ds" else v.float() for k, v in got.items()}


@pytest.mark.parametrize("kind,where", [("rank1_left_out", ("dW of encoder 2",)), ("ds_swapped", ("ds, video 3", "ds, video 4")),
                                        ("db_without_u_term", ("db of encoder 0",)), ("dQ_not_transposed", ("dQ,",))])
def test_step_bound_fails_on_each_mutation(step_self_case, kind, where):
    """The failure message names the output, the encoder and the video the mistake is in."""
    args, out = step_self_case
    got = _mutated_step(args, out, kind)
    with pytest.raises(AssertionError, match="out of bound") as e:
        _check_step(got, out)
    assert any(wh in str(e.value) for wh in where), str(e.value)


def test_ds_swap_names_the_second_video_too(step_self_case):
    args, out = step_self_case
    got = _mutated_step(args, out, "ds_swapped")
    ref, mag, depth = out["ds"]
    bad = (got["ds"].double() - ref).abs() > _bound(ref, mag, depth, torch.float32)
    assert bad[3].any() and bad[4].any() and not bad[:3].any() and not bad[5:].any()


# ---- the closed forms are the gradients (CPU, fp64 autograd through the reference modules) ---------------------------------------------
def _reference_grads_lq(P, Ws, biases, G, H, Q, Wq, Wk, ipb):
    from oracle import reference_nn as R

    B, T, K = G.shape
    E, embed = len(P), Q.shape[1]
    projs = [R.LinearProjector(p.shape[2], K).double() for p in P]
    for pr, w, b in zip(projs, Ws, biases):
        with torch.no_grad():
            pr.projector.weight.copy_(w.double())
            pr.projector.bias.copy_(b.double() if b is not None else torch.zeros(K, dtype=torch.float64))
    ad = R.CrossAttentionAdapterLearnableQuery(embed_dim=embed, llm_dim=K, token_length=T, averagetoken=True, num_encoder=E).double()
    att = ad.attention
    with torch.no_grad():
        ad.Q.copy_(Q.double())
        att.q_proj_weight.copy_(Wq.double())
        att.k_proj_weight.copy_(Wk.double())
        att.in_proj_bias.copy_(ipb.double())
    # merv.py:587-609: projector per encoder, then the adapter over the list of projected tokens
    out, w = ad([pr(p.double()) for pr, p in zip(projs, P)])
    ((out * G.double()).sum() + (w * H.double()).sum()).backward()
    grads = {"dQ": ad.Q.grad, "dWq": att.q_proj_weight.grad, "dWk": att.k_proj_weight.grad, "dbias": att.in_proj_bias.grad}
    for e, pr in enumerate(projs):
        grads[f"dW{e}"], grads[f"db{e}"] = pr.projector.weight.grad, pr.projector.bias.grad
    return grads, w.detach()


def test_closed_forms_equal_fp64_autograd_learnable_query():
    P, Ws, biases, G, _, dwo, _, Q, Wq, Wk, ipb = _step_case(**SELF_STEP, seed=9, dtype=torch.float64)
    biases = [b if b is not None else torch.zeros(SELF_STEP["K"], dtype=torch.float64) for b in biases]
    grads, w = _reference_grads_lq(P, Ws, biases, G, dwo, Q, Wq, Wk, ipb)
    embed = Q.shape[1]
    q = Wq @ Q[0] + ipb[:embed]
    u = Wk.T @ q / math.sqrt(embed)
    out, _ = closed_form_step(P, Ws, biases, G, w, dwo, u, Q, Wq, Wk, ipb)
    for name, g in grads.items():
        ref = out[name][0]
        err = float((ref.reshape(g.shape) - g).abs().max())
        assert err <= 1e-12 * max(1.0, float(g.abs().max())), (name, err)


def test_closed_forms_equal_fp64_autograd_scalar():
    from oracle import reference_nn as R

    g = torch.Generator().manual_seed(4)
    B, T, K, Cs = 5, 8, 32, (24, 16, 40, 8)  # ScalarAdapter always has four scalars
    P = [torch.rand(B, T, c, generator=g, dtype=torch.float64) + 0.2 for c in Cs]
    projs = [R.LinearProjector(c, K).double() for c in Cs]
    ad = R.ScalarAdapter().double()
    G = torch.randn(B, T, K, generator=g, dtype=torch.float64)
    H = torch.randn(1, 4, generator=g, dtype=torch.float64)
    Ys = [pr(p) for pr, p in zip(projs, P)]
    out, w = ad(Ys)
    ((out * G).sum() + (w * H).sum()).backward()
    wv = torch.softmax(ad.scalar.detach(), 0)
    gsum = G.sum(1)
    parts = [((G @ pr.projector.weight.detach()) * p).sum((1, 2))[:, None] for pr, p in zip(projs, P)]
    ref = scalar_fused_reference(wv, H[0], gsum, parts, [pr.projector.bias.detach() for pr in projs])
    tol = lambda t: 1e-12 * max(1.0, float(t.abs().max()))  # noqa: E731
    assert float((ref["dscalar"][0] - ad.scalar.grad).abs().max()) <= tol(ad.scalar.grad)
    for e, (pr, p) in enumerate(zip(projs, P)):
        assert float((ref[f"db{e}"][0] - pr.projector.bias.grad).abs().max()) <= tol(pr.projector.bias.grad)
        dW = wv[e] * G.reshape(-1, K).T @ p.reshape(-1, Cs[e])  # the GEMM of merv_wgrad_video with scale stride 0
        assert float((dW - pr.projector.weight.grad).abs().max()) <= tol(pr.projector.weight.grad)


# ---- GPU helpers --------------------------------------------------------------------------------------------------------------------
def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptrs(ts):
    from merv_b200._lib import ptr_array

    return ptr_array([0 if t is None else t.data_ptr() for t in ts])


def _sentinel(shape, dtype):
    if dtype == torch.bfloat16:
        return torch.full(shape, 0x7FA5, dtype=torch.int16, device=DEV).view(torch.bfloat16)
    return torch.full(shape, 0x7FC0ABCD, dtype=torch.int32, device=DEV).view(torch.float32)


def _is_sentinel(t):
    if t.dtype == torch.bfloat16:
        return bool((t.view(torch.int16) == 0x7FA5).all())
    return bool((t.view(torch.int32) == 0x7FC0ABCD).all())


def _split_from_workspace(lib, videos, N, C):
    parts = lib.merv_wgrad_video_parts(N, C)
    dots = -(-videos * parts // 4) * 4
    extra = lib.merv_wgrad_video_workspace(videos, N, C) - dots
    assert extra % (N * C) == 0
    return max(1, extra // (N * C)), parts


# ---- merv_wgrad_video / merv_wgrad_video_ex -----------------------------------------------------------------------------------------
# (videos, T, N_out, C, MERV_GEMM_CTA_GROUP, MERV_WGRAD_SPLIT or None): videos not divisible by the split, splits >= videos, M / N tails
WGRAD_CASES = [
    (1, 64, 8, 8, 1, None),
    (2, 128, 136, 72, 2, None),
    (5, 1024, 264, 200, 1, "3"),
    (5, 64, 264, 1032, 2, "7"),
    (33, 64, 136, 200, 1, "8"),
    (33, 128, 4096, 72, 2, "2"),
    (64, 64, 264, 768, 1, None),
    (64, 64, 136, 8, 2, "1"),
    (2, 64, 4096, 1032, 1, "2"),
    (64, 1024, 4096, 768, None, None),   # merv-full, the library's own choice: three ranges
    (64, 1024, 4096, 1024, None, None),  # merv-full: no split
]


def _set_env(monkeypatch, cta, split):
    for var, val in (("MERV_GEMM_CTA_GROUP", cta), ("MERV_WGRAD_SPLIT", split)):
        if val is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(val))


@pytest.mark.gpu
@pytest.mark.parametrize("V,T,N,C,cta,split", WGRAD_CASES)
def test_wgrad_video_meets_bounds(V, T, N, C, cta, split, monkeypatch):
    from merv_b200 import _lib, ops

    lib = _lib.load()
    _set_env(monkeypatch, cta, split)
    eff_split, parts = _split_from_workspace(lib, V, N, C)
    if split is not None:
        assert eff_split == (min(int(split), V) if int(split) > 1 else 1)
    if (V, T, N) == (64, 1024, 4096) and cta is None:
        assert eff_split == (3 if C == 768 else 1), "the library's split at the merv-full shapes changed"
    dy, x, s, w = _wgrad_case(V, T, N, C, seed=V * 7 + C, device=DEV)
    scale = torch.randn(V, 3, device=DEV)
    scale[:, 1] = s
    scale = scale[:, 1]  # strided, as weights[:, e]
    dW, partial = ops.wgrad_video(dy.reshape(V * T, N), x.reshape(V * T, C), scale, w, V)
    dW2, partial2 = ops.wgrad_video(dy.reshape(V * T, N), x.reshape(V * T, C), scale, w, V)
    torch.cuda.synchronize()
    assert torch.equal(dW, dW2) and torch.equal(partial, partial2), "not bit-reproducible run to run"
    ref, mag, dot, mdot = wgrad_reference(dy, x, s, w)
    bdw, bdot = wgrad_bounds(ref, mag, dot, mdot, T, V, eff_split, parts)
    ctas = 2 if cta == 2 else 1  # without MERV_GEMM_CTA_GROUP this kernel runs single CTAs (MN-major A: gemm_cta_group)
    check_bound(dW, ref, bdw, WgradLayout(V, eff_split, ctas))
    check_bound(partial.double().sum(1), dot, bdot, DotLayout())
    if V == 33 and split == "8":  # scale_stride 0: the scalar step's one weight for every video
        dWs, ps = ops.wgrad_video(dy.reshape(V * T, N), x.reshape(V * T, C), s[2:3].expand(V), w, V)
        ref, mag, _, _ = wgrad_reference(dy, x, s[2].expand(V), w)
        check_bound(dWs, ref, _bound(ref, mag, T + V + eff_split + 2, torch.bfloat16), WgradLayout(V, eff_split, ctas))
        assert torch.equal(ps, partial), "the dots do not depend on the scales"


@pytest.mark.gpu
@pytest.mark.parametrize("V,T,N,C,cta,split", [(5, 128, 264, 200, 2, None), (33, 64, 136, 72, 1, "3"), (64, 1024, 4096, 768, None, None)])
def test_wgrad_video_ex_reads_a_strided_slot(V, T, N, C, cta, split, monkeypatch):
    """dY read from the [:, L:L + T] slot of a NaN-filled [V, L + T + 3, N] buffer, X with ldx > C, dW written with lddw > C into a
    sentinel buffer: the block meets the bound, is bit-identical to the contiguous call and nothing around it is written."""
    from merv_b200 import _lib, ops

    lib = _lib.load()
    _set_env(monkeypatch, cta, split)
    eff_split, parts = _split_from_workspace(lib, V, N, C)
    dy, x, s, w = _wgrad_case(V, T, N, C, seed=V + C, device=DEV)
    L = 3
    buf = torch.full((V, L + T + 3, N), float("nan"), device=DEV).to(torch.bfloat16)
    slot = buf[:, L:L + T]
    slot.copy_(dy)
    xbuf = torch.full((V * T, C + 16), float("nan"), device=DEV).to(torch.bfloat16)
    xs = xbuf[:, :C]
    xs.copy_(x.reshape(V * T, C))
    dWbuf = _sentinel((N, C + 24), torch.bfloat16)
    partial = torch.empty((V, CHUNKS), device=DEV)
    ws = torch.empty(max(int(lib.merv_wgrad_video_workspace(V, N, C)), 4), device=DEV)
    _lib.check(lib.merv_wgrad_video_ex(slot.data_ptr(), slot.stride(1), slot.stride(0), xs.data_ptr(), xs.stride(0), s.data_ptr(), 1, w.data_ptr(),
                                       w.stride(0), dWbuf.data_ptr(), dWbuf.stride(0), partial.data_ptr(), ws.data_ptr(), V, T, N, C, _stream()))
    want, want_p = ops.wgrad_video(dy.reshape(V * T, N), x.reshape(V * T, C), s, w, V)
    torch.cuda.synchronize()
    assert _is_sentinel(dWbuf[:, C:]), "merv_wgrad_video_ex wrote past column C of a wider dW"
    assert torch.equal(dWbuf[:, :C], want) and torch.equal(partial, want_p), "the strided form differs from the contiguous one"
    ref, mag, dot, mdot = wgrad_reference(dy, x, s, w)
    bdw, bdot = wgrad_bounds(ref, mag, dot, mdot, T, V, eff_split, parts)
    check_bound(dWbuf[:, :C], ref, bdw, WgradLayout(V, eff_split, 2 if cta == 2 else 1))
    check_bound(partial.double().sum(1), dot, bdot, DotLayout())


# ---- merv_video_colsum / merv_colsum ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("T", [1, 31, 32, 96, 97, 128, 129, 1024])
def test_video_colsum_meets_bound(dtype, T):
    from merv_b200 import ops

    B = 3
    vec = 8 if dtype == torch.bfloat16 else 4
    for K in ((8, 72, 200, 4096) if dtype == torch.bfloat16 else (4, 12, 200)):
        g = torch.Generator().manual_seed(T * 10 + K)
        pad = 2 * vec  # ld > K, and batch_stride > T * ld (the videos are a slot of a longer buffer)
        buf = (torch.randn(B, T + 5, K + pad, generator=g) + 0.3).to(dtype).to(DEV)
        x = buf[:, 2:2 + T, :K]
        for scale in (1.0, 0.37):
            got = ops.video_colsum(x, scale)
            x64 = x.double()
            ref, mag = scale * x64.sum(1), scale * x64.abs().sum(1)
            # ceil(T / 32) adds per thread, the 32 row groups in order, the scale
            check_bound(got, ref, 4 * U * (math.ceil(T / 32) + 32 + 1) * mag, VideoLayout(("column",)))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("M,N", [(77, 200), (256, 72), (600, 4096), (1000, 100), (300, 13)])
def test_colsum_meets_bound(dtype, M, N):
    """M < 256, whole and partial 256-row blocks; N not a multiple of the vector width takes the scalar kernels."""
    from merv_b200 import ops

    g = torch.Generator().manual_seed(M + N)
    x = (torch.randn(M, N + 8, generator=g) + 0.3).to(dtype).to(DEV)[:, :N]
    got = ops.colsum(x)
    ref, mag = x.double().sum(0), x.double().abs().sum(0)
    vec = 8 if dtype == torch.bfloat16 else 4
    # stage 1 per 256-row block: the vector path (N and ld whole vectors) adds 256 / 32 rows per thread, then its 32 row groups in order;
    # the scalar path adds the block's 256 rows in order.  Stage 2 adds the ceil(M / 256) block sums in order.
    stage1 = 256 // 32 + 32 if N % vec == 0 and x.stride(0) % vec == 0 else 256
    check_bound(got, ref, _bound(ref, mag, stage1 + -(-M // 256), dtype), OutLayout("colsum", ("column",)))


# ---- merv_pair_dot / merv_pair_dot_scale -----------------------------------------------------------------------------------------
def _pair_dot_cases():
    out = []
    for dtype, vec in ((torch.bfloat16, 8), (torch.float32, 4)):
        edge = 32 * 256 * vec
        for B, n in ((1, 8), (3, 248), (64, edge - vec), (3, edge + vec), (64, edge + vec), (3, 1 << 21)):
            out.append((dtype, B, n))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,B,n", _pair_dot_cases())
def test_pair_dot_meets_bound_per_chunk(dtype, B, n):
    from merv_b200 import ops

    vec = 8 if dtype == torch.bfloat16 else 4
    g = torch.Generator().manual_seed(B * 31 + n)
    x = (torch.randn(B, n, generator=g) + 0.2).to(dtype).to(DEV)
    y = (torch.randn(B, n, generator=g) - 0.1).to(dtype).to(DEV)
    sfull = torch.randn(B, 3, generator=g).to(DEV)
    scale = sfull[:, 1]
    part = ops.pair_dot(x, y)
    part2, ys = ops.pair_dot(x, y, scale=scale)
    torch.cuda.synchronize()
    assert torch.equal(part, part2)
    assert torch.equal(ys, (y.float() * scale[:, None]).to(dtype)), "y_scaled is not one fp32 multiply and one rounding"
    nvec = n // vec
    per = -(-nvec // CHUNKS)
    prod = torch.zeros(B, CHUNKS * per * vec, dtype=torch.float64, device=DEV)
    prod[:, :n] = x.double() * y.double()
    ref = prod.view(B, CHUNKS, per * vec).sum(-1)
    mag = prod.abs().view(B, CHUNKS, per * vec).sum(-1)
    empty = torch.arange(CHUNKS, device=DEV) * per >= nvec
    assert (part[:, empty] == 0).all(), "an empty chunk is not exactly 0"
    # a thread's fma chain covers at most ceil(per / 256) vectors of its chunk, then the 256-thread block sum (two 5-level warp trees)
    depth = math.ceil(per / 256) * vec + 10
    check_bound(part, ref, 4 * U * depth * mag, DotLayout())
    check_bound(part.double().sum(1), ref.sum(1), 4 * U * depth * mag.sum(1), DotLayout())


# ---- merv_transpose_rowscale ----------------------------------------------------------------------------------------------------------
# (dtype, R, C, rows_per_scale, ldx extra, R_pad extra, ldy extra): the first two take the 16-byte bf16 kernel; the next two the scalar
# kernel in bf16 (C % 8 != 0, then ldx % 8 != 0); the last two the scalar kernel in fp32
TRANSPOSE_CASES = [
    (torch.bfloat16, 231, 200, 77, 8, 1, 8),
    (torch.bfloat16, 128, 64, 64, 0, 0, 16),
    (torch.bfloat16, 135, 74, 27, 2, 1, 4),
    (torch.bfloat16, 40, 16, 1, 2, 0, 8),
    (torch.float32, 154, 12, 77, 4, 2, 4),
    (torch.float32, 64, 200, 1, 0, 0, 3),
]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,R,C,rps,xe,pe,ye", TRANSPOSE_CASES)
def test_transpose_rowscale_is_bit_identical(dtype, R, C, rps, xe, pe, ye):
    from merv_b200 import _lib, ops

    lib = _lib.load()
    vec = 8 if dtype == torch.bfloat16 else 4
    Rp = (-(-R // vec) * vec if pe else R) + (vec if pe and R % vec == 0 else 0)
    g = torch.Generator().manual_seed(R + C)
    x = torch.randn(R, C + xe, generator=g).to(dtype).to(DEV)[:, :C]
    nsc = -(-R // rps)
    sfull = torch.randn(nsc, 2, generator=g).to(DEV)
    for scale in (sfull[:, 1], None):
        y = _sentinel((C, Rp + ye), dtype)
        _lib.check(lib.merv_transpose_rowscale(x.data_ptr(), y.data_ptr(), R, Rp, C, x.stride(0), y.stride(0), None if scale is None else scale.data_ptr(), 0 if scale is None else scale.stride(0), rps, ops.dtype_code(dtype), _stream()))
        torch.cuda.synchronize()
        want = x if scale is None else (x.float() * scale.repeat_interleave(rps)[:R, None]).to(dtype)
        assert torch.equal(y[:, :R], want.T), f"scale={'none' if scale is None else 'strided'}: not bit-identical to torch"
        assert Rp == R or bool((y[:, R:Rp] == 0).all()) and not bool(torch.signbit(y[:, R:Rp].float()).any()), "the pad is not exactly +0"
        assert _is_sentinel(y[:, Rp:]), "wrote past R_pad"


# ---- the two-GEMM form (T % 64 != 0) -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cta", [1, 2])
@pytest.mark.parametrize("B,T,K,C", [(3, 77, 264, 200), (5, 77, 4096, 72), (2, 27, 136, 1032)])
def test_two_gemm_form_meets_bound(B, T, K, C, cta, monkeypatch):
    from merv_b200 import ops
    from tests.test_fused_forward_kernels import gemm_reference

    monkeypatch.setenv("MERV_GEMM_CTA_GROUP", str(cta))
    g = torch.Generator().manual_seed(B * T + K + C)
    G = (torch.randn(B * T, K, generator=g) + 0.1).to(torch.bfloat16).to(DEV)
    W = ((torch.rand(K, C, generator=g) - 0.3) / math.sqrt(C)).to(torch.bfloat16).to(DEV)
    Ps = (torch.rand(B * T, C, generator=g) + 0.1).to(torch.bfloat16).to(DEV)
    one = torch.ones((1, 1), device=DEV)
    Z = ops.gemm_ex(G, W, w_t=True)  # dOut W_e
    ref, mag = gemm_reference([G], [W.T], one, None, B * T)
    check_bound(Z, ref, gemm_bound(ref, mag, [K]), GemmLayout(T))
    dW = ops.gemm_ex(G, Ps, a_t=True, w_t=True)  # dOut^T (w_e (.) P_e), contraction over B * T tokens
    ref, mag = gemm_reference([G.T], [Ps.T], one, None, K)
    check_bound(dW, ref, gemm_bound(ref, mag, [B * T]), GemmLayout(K))


# ---- merv_fused_backward -----------------------------------------------------------------------------------------------------------
# name: (dtype, B, C per encoder, K, embed, options); options: "nobias" encoders, "db_null" encoders (bias kept), "dwo", "ipb", "wide"
FBWD_CASES = {
    "bf16_e1_k8": (torch.bfloat16, 1, (64,), 8, 8, dict(dwo=True, ipb=True)),
    "bf16_e2_k100": (torch.bfloat16, 5, (200, 72), 100, 40, dict(nobias=(1,), dwo=False, ipb=True)),
    "bf16_e3_c12_b33": (torch.bfloat16, 33, (136, 12, 64), 256, 48, dict(db_null=(0,), dwo=True, ipb=False)),
    "bf16_e4_full": (torch.bfloat16, 64, (1024, 1024, 768, 768), 4096, 3072, dict(dwo=True, ipb=True)),
    "bf16_e8_wide": (torch.bfloat16, 64, (8, 16, 24, 200, 72, 136, 64, 8), 264, 48, dict(nobias=(2, 5), db_null=(6,), dwo=True, ipb=True, wide=True)),
    "f32_e2_c6": (torch.float32, 5, (200, 6), 100, 40, dict(dwo=True, ipb=True)),
    "f32_e8_wide": (torch.float32, 33, (4, 8, 12, 200, 72, 136, 64, 16), 256, 48, dict(nobias=(0,), db_null=(3,), dwo=False, ipb=False, wide=True)),
    "f32_e3_k4096": (torch.float32, 1, (128, 64, 200), 4096, 3072, dict(dwo=True, ipb=True)),
}


def _fbwd_inputs(name):
    dt, B, Cs, K, embed, o = FBWD_CASES[name]
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    E = len(Cs)
    on = lambda t: t.to(DEV)  # noqa: E731
    scores = torch.randn(B, E, generator=g) + torch.remainder(torch.arange(B)[:, None] * 3 + torch.arange(E)[None], 5) * 0.4
    weights = on(torch.softmax(scores, -1).float())
    dwo = on(torch.randn(B, E, generator=g) * 2) if o.get("dwo") else None
    u = on(torch.randn(K, generator=g) * 0.5)
    gsum = on(torch.randn(B, K, generator=g) * 3 + 0.5)
    parts = [on(torch.randn(B, CHUNKS, generator=g) * 0.5 + 0.2 * (e - 1)) for e in range(E)]
    pbar = [on(torch.rand(B, c, generator=g) + 0.2) for c in Cs]
    pad = 8 if o.get("wide") else 0
    Ws, dW_in, dW_views, biases = [], [], [], []
    for e, c in enumerate(Cs):
        wbuf = torch.full((K, c + pad), float("nan")).to(dt)  # columns past C_e must never be read
        wbuf[:, :c] = ((torch.rand(K, c, generator=g) - 0.3) / math.sqrt(c)).to(dt)
        Ws.append(on(wbuf)[:, :c])
        dW_in.append(on((torch.randn(K, c, generator=g) * 0.5).to(dt)))
        biases.append(None if e in o.get("nobias", ()) else on((torch.randn(K, generator=g) * 0.5).to(dt)))
    Q = on(torch.randn(1, embed, generator=g).to(dt))
    Wq = on((torch.randn(embed, embed, generator=g) / math.sqrt(embed)).to(dt))
    Wk = on((torch.randn(embed, K, generator=g) / math.sqrt(embed)).to(dt))
    ipb = on((torch.randn(3 * embed, generator=g) * 0.3).to(dt)) if o.get("ipb") else None
    return dt, o, weights, dwo, u, gsum, parts, pbar, Ws, biases, Q, Wq, Wk, ipb, dW_in


def run_fused_backward(dt, weights, dwo, u, gsum, parts, pbar, Ws, biases, Q, Wq, Wk, ipb, dWs, lddw, db_null=()):
    """merv_fused_backward through its descriptor (as ops.fused_backward fills it), with the db entries of `db_null` NULL."""
    from merv_b200 import _lib, ops

    lib = _lib.load()
    B, E = weights.shape
    K, embed = u.numel(), Wk.shape[0]
    d = _lib.FusedBwdDesc()
    d.B, d.E, d.K, d.embed = B, E, K, embed
    ds = torch.empty((B, E), device=DEV)
    dbs = [None if (b is None or e in db_null) else torch.empty(K, dtype=dt, device=DEV) for e, b in enumerate(biases)]
    dQ, dWq = torch.empty((1, embed), dtype=dt, device=DEV), torch.empty((embed, embed), dtype=dt, device=DEV)
    dWk, dbias = torch.empty((embed, K), dtype=dt, device=DEV), torch.empty(3 * embed, dtype=dt, device=DEV)
    for e in range(E):
        d.C[e] = Ws[e].shape[1]
        d.dw_partial[e], d.pbar[e] = parts[e].data_ptr(), pbar[e].data_ptr()
        d.W[e], d.ldw[e], d.bias[e] = Ws[e].data_ptr(), Ws[e].stride(0), None if biases[e] is None else biases[e].data_ptr()
        d.dW[e], d.lddw[e], d.db[e] = dWs[e].data_ptr(), lddw[e], None if dbs[e] is None else dbs[e].data_ptr()
    d.weights, d.dweights_out, d.u, d.gsum = weights.data_ptr(), None if dwo is None else dwo.data_ptr(), u.data_ptr(), gsum.data_ptr()
    d.Q, d.Wq, d.Wk, d.in_proj_bias = Q.data_ptr(), Wq.data_ptr(), Wk.data_ptr(), None if ipb is None else ipb.data_ptr()
    d.ds, d.dQ, d.dWq, d.dWk, d.dbias = ds.data_ptr(), dQ.data_ptr(), dWq.data_ptr(), dWk.data_ptr(), dbias.data_ptr()
    n = lib.merv_fused_backward_workspace(ctypes.byref(d))
    ws = torch.empty(max(n, 1), device=DEV)
    d.workspace, d.workspace_floats = ws.data_ptr(), n
    _lib.check(lib.merv_fused_backward(ctypes.byref(d), ops.dtype_code(dt), _stream()))
    torch.cuda.synchronize()
    return ds, dbs, dQ, dWq, dWk, dbias


def check_fused_backward(dt, got, ref, E, dbs_expected, eps=0.0, gemm_parts=None):
    """Every output of merv_fused_backward per element; dbias[embed:] exactly 0."""
    ds, dWs, dbs, dQ, dWq, dWk, dbias = got
    r, m, n = ref["ds"]
    check_bound(ds, r, _bound(r, m, n, torch.float32, eps), OutLayout("ds", ("video", "encoder")))
    for e in range(E):
        r, m, n = ref[f"dW{e}"]
        b = _bound(r, m, n, dt, eps)
        if gemm_parts is not None:  # the GEMM's own bf16 rounding of dOut^T (w_e (.) P_e)
            b = b + BF16_REL * gemm_parts[e].abs()
        check_bound(dWs[e], r, b, OutLayout("dW", ("row", "column"), e))
        if dbs_expected[e]:
            r, m, n = ref[f"db{e}"]
            check_bound(dbs[e], r, _bound(r, m, n, dt, eps), OutLayout("db", ("row",), e))
        else:
            assert dbs[e] is None
    embed = dQ.shape[1]
    for name, t in (("dQ", dQ), ("dWq", dWq), ("dWk", dWk)):
        r, m, n = ref[name]
        check_bound(t, r, _bound(r, m, n, dt, eps), OutLayout(name, ("row", "column")))
    r, m, n = ref["dbias"]
    check_bound(dbias[:embed], r[:embed], _bound(r[:embed], m[:embed], n, dt, eps), OutLayout("dbias", ("element",)))
    assert bool((dbias[embed:] == 0).all()), "the k / v parts of the in_proj_bias gradient are not exactly 0"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FBWD_CASES))
def test_fused_backward_meets_bounds(name):
    dt, o, weights, dwo, u, gsum, parts, pbar, Ws, biases, Q, Wq, Wk, ipb, dW_in = _fbwd_inputs(name)
    E, K = len(Ws), u.numel()
    pad = 16 if o.get("wide") else 0
    bufs = [_sentinel((K, w.shape[1] + pad), dt) for w in Ws]
    for buf, d0 in zip(bufs, dW_in):
        buf[:, :d0.shape[1]] = d0
    dWs = [buf[:, :w.shape[1]] for buf, w in zip(bufs, Ws)]
    db_null = o.get("db_null", ())
    ds, dbs, dQ, dWq, dWk, dbias = run_fused_backward(dt, weights, dwo, u, gsum, parts, pbar, Ws, biases, Q, Wq, Wk, ipb, dWs,
                                                       [b.stride(0) for b in bufs], db_null)
    for e, buf in enumerate(bufs):
        assert pad == 0 or _is_sentinel(buf[:, Ws[e].shape[1]:]), f"encoder {e}: dW written past column C_e"
    absm = lambda t: (t.double(), t.double().abs())  # noqa: E731
    ref = fused_bwd_reference(weights, dwo, u, absm(gsum), [absm(p) for p in parts], [absm(p) for p in pbar], Ws, biases, Q, Wq, Wk, ipb,
                              [(d.double(), torch.zeros_like(d, dtype=torch.float64)) for d in dW_in])
    check_fused_backward(dt, (ds, dWs, dbs, dQ, dWq, dWk, dbias), ref, E, [b is not None and e not in db_null for e, b in enumerate(biases)])


# ---- merv_scalar_fused_backward ----------------------------------------------------------------------------------------------------
SCALAR_CASES = [(1, 1, 8), (2, 33, 100), (3, 0, 256), (4, 33, 257), (5, 1, 4096), (8, 33, 4096), (8, 0, 100), (6, 33, 257)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("E,B,K", SCALAR_CASES)
def test_scalar_fused_backward_meets_bounds(E, B, K, dtype):
    from merv_b200 import _lib, ops

    lib = _lib.load()
    g = torch.Generator().manual_seed(E * 100 + B + K)
    on = lambda t: t.to(DEV)  # noqa: E731
    w = on(torch.softmax(torch.randn(E, generator=g), 0).float())
    dwo = None if (E + B) % 2 else on(torch.randn(E, generator=g) * 2)
    gsum = on(torch.randn(B, K, generator=g) + 0.3)
    parts = [on(torch.randn(B, CHUNKS, generator=g) * 0.5 + 0.1 * e) for e in range(E)]
    biases = [None if e % 3 == 1 else on((torch.randn(K, generator=g) * 0.5).to(dtype)) for e in range(E)]
    db_null = {e for e in range(E) if e % 4 == 2}  # a NULL db next to a present bias
    dbs = [None if (b is None or e in db_null) else torch.empty(K, dtype=dtype, device=DEV) for e, b in enumerate(biases)]
    dscalar = torch.empty(E, device=DEV)
    n = lib.merv_scalar_fused_backward_workspace(E, K)
    ws = torch.empty(max(n, 1), device=DEV)
    _lib.check(lib.merv_scalar_fused_backward(w.data_ptr(), None if dwo is None else dwo.data_ptr(), gsum.data_ptr() if B else None, _ptrs(parts),
                                              _ptrs(biases), _ptrs(dbs), dscalar.data_ptr(), ws.data_ptr(), n, B, E, K, ops.dtype_code(dtype),
                                              _stream()))
    torch.cuda.synchronize()
    ref = scalar_fused_reference(w, dwo, gsum, parts, biases)
    r, m, depth = ref["dscalar"]
    check_bound(dscalar, r, _bound(r, m, depth, torch.float32) + TINY, OutLayout("dscalar", ("encoder",)))
    for e in range(E):
        if dbs[e] is not None:
            r, m, depth = ref[f"db{e}"]
            check_bound(dbs[e], r, _bound(r, m, depth, dtype), OutLayout("db", ("row",), e))


# ---- the chain: each fused step composed by hand from the calls its backward makes ------------------------------------------------------
def hand_step(P, Ws, biases, G, weights, dwo, u, Q, Wq, Wk, ipb):
    """The backward of _FusedLinearFn (merv_b200/nn_utils.py) from its ops calls: merv_wgrad_video when T % 64 == 0, else Z_e = dOut W_e,
    merv_pair_dot_scale and dOut^T (w_e (.) P_e); merv_video_colsum; merv_fused_backward."""
    from merv_b200 import ops

    B, T, K = G.shape
    g = G.reshape(B * T, K)
    gsum = ops.video_colsum(G)
    parts, pbars, dWs = [], [], []
    for e, p in enumerate(P):
        Pe = p.reshape(B * T, -1)
        if T % 64 == 0:
            dW, dwp = ops.wgrad_video(g, Pe, weights[:, e], Ws[e], B)
        else:
            Z = ops.gemm_ex(g, Ws[e], w_t=True)
            dwp, Ps = ops.pair_dot(Z.reshape(B, -1), Pe.reshape(B, -1), scale=weights[:, e])
            dW = ops.gemm_ex(g, Ps.view(B * T, -1), a_t=True, w_t=True)
        parts.append(dwp)
        pbars.append(ops.video_colsum(p, 1.0 / T))
        dWs.append(dW)
    ds, dbs, dQ, dWq, dWk, dbias = ops.fused_backward(weights, dwo, u, gsum, parts, pbars, Ws, biases, Q, Wq, Wk, ipb, dWs)
    torch.cuda.synchronize()
    return ds, dWs, dbs, dQ, dWq, dWk, dbias


def hand_scalar_step(P, Ws, biases, G, w, dwo):
    """The backward of _FusedScalarLinearFn (merv_b200/nn_utils.py) from its ops calls: merv_wgrad_video with scale stride 0 per encoder,
    merv_video_colsum, merv_scalar_fused_backward.  Returns (dscalar, [dW_e], [db_e])."""
    from merv_b200 import ops

    B, T, K = G.shape
    g = G.reshape(B * T, K)
    gsum = ops.video_colsum(G)
    dWs, parts = [], []
    for e, p in enumerate(P):
        dW, dwp = ops.wgrad_video(g, p.reshape(B * T, -1), w[e].expand(B), Ws[e], B)
        dWs.append(dW)
        parts.append(dwp)
    dscalar, dbs = ops.scalar_fused_backward(w, dwo, gsum, parts, biases)
    torch.cuda.synchronize()
    return dscalar, dWs, dbs


def _stage1_eps(lib, B, T, K, Cs):
    """Relative error (to their mags) of the quantities a whole step feeds its last kernel: with T % 64 == 0 the dots, gsum, pbar and the
    GEMM part of dW come from one accumulator per video, its epilogue and the folds; otherwise Z_e = dOut W_e and w_e (.) P_e are stored in
    bf16 before they are reduced."""
    if T % 64 == 0:
        parts = max(lib.merv_wgrad_video_parts(K, c) for c in Cs)
        return 4 * U * (T + B + EPI_COLS + WARP_LEVELS + math.ceil(parts / CHUNKS) + 10)
    return BF16_REL + 4 * U * (K + B * T + 64)


# name: (B, T, C per encoder, K, embed)
CHAIN_CASES = {
    "t64_e2": (5, 64, (200, 72), 264, 48),
    "t128_e4_b33": (33, 128, (136, 64, 8, 200), 264, 40),
    "t77_e3": (3, 77, (200, 72, 136), 264, 48),
    "t77_e2_b33": (33, 77, (72, 64), 136, 40),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CHAIN_CASES))
def test_fused_step_meets_closed_form_bounds(name):
    from merv_b200 import _lib

    lib = _lib.load()
    B, T, Cs, K, embed = CHAIN_CASES[name]
    args = _step_case(B, T, Cs, K, embed, seed=sum(map(ord, name)), device=DEV)
    P, Ws, biases, G, weights, dwo, u, Q, Wq, Wk, ipb = args
    got = hand_step(*args)
    again = hand_step(*args)
    for a, b in zip(got, again):
        for x, y in zip(a if isinstance(a, list) else [a], b if isinstance(b, list) else [b]):
            assert (x is None and y is None) or torch.equal(x, y), "the step is not bit-reproducible"
    out, gemm = closed_form_step(*args)
    eps = _stage1_eps(lib, B, T, K, Cs)
    check_fused_backward(torch.bfloat16, got, out, len(Cs), [b is not None for b in biases], eps=eps, gemm_parts=gemm)


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,Cs,K", [(5, 64, (200, 72, 136, 64), 264), (33, 128, (72, 8), 136)])
def test_fused_scalar_step_meets_closed_form_bounds(B, T, Cs, K):
    """_FusedScalarLinearFn's backward from its ops calls: merv_wgrad_video with scale stride 0, merv_video_colsum, merv_scalar_fused_backward."""
    from merv_b200 import _lib, ops

    lib = _lib.load()
    P, Ws, biases, G, _, dwo, _, _, _, _, _ = _step_case(B, T, Cs, K, 8, seed=B + T, device=DEV)
    E = len(Cs)
    w = torch.softmax(torch.arange(E, dtype=torch.float32, device=DEV) * 0.3 - 0.4, 0)
    dwo = dwo[0, :E].contiguous()
    dscalar, dWs, dbs = hand_scalar_step(P, Ws, biases, G, w, dwo)
    G64 = G.double()
    pm = [(((G64 @ W.double()) * p.double()).sum((1, 2))[:, None], ((G64.abs() @ W.double().abs()) * p.double().abs()).sum((1, 2))[:, None])
          for W, p in zip(Ws, P)]
    ref = scalar_fused_reference(w, dwo, (G64.sum(1), G64.abs().sum(1)), pm, biases)
    eps = _stage1_eps(lib, B, T, K, Cs)
    r, m, depth = ref["dscalar"]
    check_bound(dscalar, r, _bound(r, m, depth, torch.float32, eps), OutLayout("dscalar", ("encoder",)))
    for e in range(E):
        if biases[e] is not None:
            r, m, depth = ref[f"db{e}"]
            check_bound(dbs[e], r, _bound(r, m, depth, torch.bfloat16, eps), OutLayout("db", ("row",), e))
        ref_w, mag_w, _, _ = wgrad_reference(G.view(B, T, K), P[e], w[e].expand(B), Ws[e])
        check_bound(dWs[e], ref_w, _bound(ref_w, mag_w, T + B + 8 + 2, torch.bfloat16), OutLayout("dW", ("row", "column"), e))


# ---- the modules' own backward is the hand composition, bit for bit -----------------------------------------------------------------------
def _function_node(t, name):
    """The autograd node of the custom Function `name` behind tensor t."""
    stack, seen = [t.grad_fn], set()
    while stack:
        n = stack.pop()
        if n is None or id(n) in seen:
            continue
        seen.add(id(n))
        if type(n).__name__ == name + "Backward":
            return n
        stack += [f for f, _ in n.next_functions]
    raise AssertionError(f"the training step did not run through {name}")


def _fused_module(mixer, Cs, K, embed, T, frames, S, seed):
    """MervFusion(3d-avg pool + Linear projectors, linked mixer, fused_training=True) in bf16, train mode, as MERV trains it."""
    import merv_b200 as M

    torch.manual_seed(seed)
    projs = [M.AveragePooling3DProjector(C, K, frames, S, "linear") for C in Cs]
    if mixer == "lq":
        ff = M.CrossAttentionAdapterLearnableQuery(embed, K, T, averagetoken=True, num_encoder=len(Cs))
        with torch.no_grad():
            ff.Q.mul_(8.0)  # a mixing softmax far from uniform
            ff.attention.in_proj_bias.normal_(0.0, 0.3)
    else:
        ff = M.ScalarAdapter(len(Cs))
    return M.MervFusion(projs, ff, fused_training=True).to(device=DEV, dtype=torch.bfloat16).train()


def _module_step(m, B, Fin, H, Cs, seed, fn):
    """Features with a distinct mean per encoder, forward, backward of sum(G * out) + sum(Hw * weights); returns (the tensors the Function
    `fn` saved, read before the backward frees them, G, Hw)."""
    g = torch.Generator().manual_seed(seed)
    xs = [(torch.randn(B, Fin, H * H, c, generator=g) + 0.4 * (e - 1)).to(torch.bfloat16).to(DEV) for e, c in enumerate(Cs)]
    m.zero_grad(set_to_none=True)
    out, w = m(xs)
    saved = _function_node(out, fn).saved_tensors
    G = (torch.randn(out.shape, generator=g) * 0.5 + 0.1).to(torch.bfloat16).to(DEV)
    Hw = (torch.randn(w.shape, generator=g) * 4).to(torch.bfloat16).to(DEV)
    torch.autograd.backward([out, w], [G, Hw])
    torch.cuda.synchronize()
    return saved, G, Hw


def _assert_grad(param, want, what):
    assert param.grad is not None, f"{what}: no gradient"
    assert torch.equal(param.grad, want.reshape(param.shape).to(param.dtype)), f"{what}: the module's gradient differs from the hand composition"


# name: (B, input frames, patch grid side, output frames, pooled side S, channels per encoder, K, embed); T = output frames * S^2
MODULE_CASES = {
    "t64": (5, 8, 8, 4, 4, (64, 136, 200), 264, 48),
    "t128_b33": (33, 8, 8, 8, 4, (72, 64), 136, 40),
    "t27_two_gemm": (3, 6, 7, 3, 3, (200, 72, 136), 264, 48),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MODULE_CASES))
def test_fused_training_gradients_are_the_hand_composition(name):
    """MervFusion(fused_training=True) with the learnable-query mixer: every parameter gradient is bit-identical to hand_step on the tensors
    the Function saved (pooled tokens, fp32 weights, u, bf16 parameters) and the same dOut / dweights.  This pins the glue of
    _FusedLinearFn.backward (the dOut view, the weights[:, e] scales, the dweights cast, the order of the returned gradients, their dtype);
    the gradients then meet the fp64 closed-form bounds."""
    from merv_b200 import _lib

    B, Fin, H, frames, S, Cs, K, embed = MODULE_CASES[name]
    T = frames * S * S
    m = _fused_module("lq", Cs, K, embed, T, frames, S, seed=sum(map(ord, name)))
    saved, G, Hw = _module_step(m, B, Fin, H, Cs, len(name), "_FusedLinearFn")
    E = len(Cs)
    weights, u, Qc, Wqc, Wkc, bc = saved[:6]
    pooled, Ws, biases = saved[6:6 + E], saved[6 + E:6 + 2 * E], saved[6 + 2 * E:6 + 3 * E]
    P = [p.reshape(B, T, -1) for p in pooled]
    G3 = G.reshape(B, T, K)
    args = (P, list(Ws), list(biases), G3, weights, Hw.float(), u, Qc, Wqc, Wkc, bc)
    got = hand_step(*args)
    ds, dWs, dbs, dQ, dWq, dWk, dbias = got
    ff, att = m.feature_fusion, m.feature_fusion.attention
    _assert_grad(ff.Q, dQ, "Q")
    _assert_grad(att.q_proj_weight, dWq, "q_proj_weight")
    _assert_grad(att.k_proj_weight, dWk, "k_proj_weight")
    _assert_grad(att.in_proj_bias, dbias, "in_proj_bias")
    for e, proj in enumerate(m.projectors):
        lin = proj.layers()[0][0]
        _assert_grad(lin.weight, dWs[e], f"projector {e} weight")
        _assert_grad(lin.bias, dbs[e], f"projector {e} bias")
    ref, gemm = closed_form_step(*args)
    check_fused_backward(torch.bfloat16, got, ref, E, [True] * E, eps=_stage1_eps(_lib.load(), B, T, K, Cs), gemm_parts=gemm)


@pytest.mark.gpu
@pytest.mark.parametrize("B,frames", [(5, 4), (33, 8)])
def test_fused_scalar_training_gradients_are_the_hand_composition(B, frames):
    """MervFusion(fused_training=True) with the scalar mixer (four encoders: the mixer always holds four scalars): the scalar and every
    projector gradient are bit-identical to hand_scalar_step on the tensors _FusedScalarLinearFn saved."""
    Cs, K, S = (64, 136, 200, 72), 264, 4
    T = frames * S * S
    m = _fused_module("scalar", Cs, K, 0, T, frames, S, seed=B)
    (w32, *saved), G, Hw = _module_step(m, B, 8, 8, Cs, B + 1, "_FusedScalarLinearFn")
    E = len(Cs)
    pooled, Ws, biases = saved[:E], saved[E:2 * E], saved[2 * E:3 * E]
    dscalar, dWs, dbs = hand_scalar_step([p.reshape(B, T, -1) for p in pooled], list(Ws), list(biases), G.reshape(B, T, K), w32,
                                         Hw.float().reshape(-1).contiguous())
    _assert_grad(m.feature_fusion.scalar, dscalar, "scalar")
    for e, proj in enumerate(m.projectors):
        lin = proj.layers()[0][0]
        _assert_grad(lin.weight, dWs[e], f"projector {e} weight")
        _assert_grad(lin.bias, dbs[e], f"projector {e} bias")
