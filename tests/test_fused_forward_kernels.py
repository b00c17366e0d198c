"""The kernels of the fused forward chain, called directly and compared element by element with fp64 references.

`merv_fused_forward` is pool -> scores + softmax -> fused projector+mix GEMM.  Each piece is tested here on its own, at the shapes where
tiling and scheduling go wrong (ragged K, N tails inside an output box, videos that straddle a 128-row tile, capped persistent grids,
strided outputs), and the whole chain is compared bit for bit with its own three-launch composition.

Every reference is computed in fp64 from the inputs the kernel was actually given (bf16 operands are already rounded), and every check
is per element: ``check_bound(got, ref, bound, layout)`` asserts ``|got - ref| <= bound`` and names the worst element in kernel terms
(video, row in the video, column, 128 x 256 tile, output box or segment).  A global ``max|a-b| / max|b|`` would not see a video given
its neighbour's weight, a dropped K tail or a bias row taken from the wrong video.

Error model, with u = 2^-24 (fp32 unit roundoff) and ``mag`` the reference expression with every term replaced by its absolute value:

* fused GEMM, ``ref = sum_s scale[v, s] (A_s W_s^T)[m] + bias_mix[v]``:
  ``bound = 2^-8 |ref| + 4 u (sum_s K_s + E) mag``.  The first term is the bf16 rounding of the output (at most half a bf16 ulp,
  2^-9 |ref|, doubled for the value the rounding starts from), the second the fp32 accumulation: K_s products per segment on the tensor
  cores, then E scaled segment sums and the bias in the epilogue, each addition off by at most a few u of the running magnitude.
* scores, ``s = (1/T) sum_i p_i + c``: each thread sums ceil(count / 256) partials, then a 5-level warp tree and a 5-level block tree,
  then the division and the constant: ``bound = (ceil(count / 256) + 12) u (sum|p| / T + |c|)``.
* weights, ``w = softmax(s)`` of the fp32 scores: expf is within 2 ulp (4 u relative), ``s - max`` is rounded (u |s - max| relative after
  the exponential), the denominator adds the same relative errors plus at most 3 tree additions and the (E - 1)/e of its own rounded
  arguments, and the division is correctly rounded: ``bound = (16 + |s - max|) u w + 2^-126`` (the last term covers exponentials that
  underflow).  The weights sum to 1 within E u, since numerators and denominator share their exponentials, and E = 1 gives exactly 1.0.
* ``bias_mix = sum_e w_e b_e`` with the kernel's own fp32 weights: E fused multiply-adds, ``bound = (E + 1) u sum_e w_e |b_e|``.
* ``softmax_mix``, ``out = sum_e w_e V_e`` with the kernel's own weights: ``(E + 1) u sum_e w_e |V_e|``, plus ``2^-8 |ref|`` for bf16.

The CPU tests below show that this harness catches the mistakes it is meant to catch, by feeding it the bf16-rounded reference with
one deliberate mutation at a time.
"""
import math

import pytest
import torch
import torch.nn.functional as F

DEV = "cuda:0"
U = 2.0 ** -24
BF16_REL = 2.0 ** -8
TINY = 2.0 ** -126
TILE_M, TILE_N, BOX_N = 128, 256, 32


# ---- the harness ----------------------------------------------------------------------------------------------------------------------
class GemmLayout:
    """Names an element of a [M, N] GEMM output (or of a [B, rows_per_video, N] view of it) in kernel terms."""

    def __init__(self, rows_per_video):
        self.rows_per_video = rows_per_video

    def describe(self, idx):
        if len(idx) == 3:
            b, r, n = idx
            m = b * self.rows_per_video + r
        else:
            m, n = idx
        return (f"video {m // self.rows_per_video}, row {m % self.rows_per_video} of the video, column {n}, "
                f"{TILE_M}x{TILE_N} tile (row block {m // TILE_M}, column block {n // TILE_N}), {BOX_N}-column output box {n // BOX_N}")


class VideoLayout:
    """[B, E] (scores, weights: segment = encoder), [B, N] (bias_mix) or [B, T, K] (mixed tokens)."""

    def __init__(self, inner=("segment",)):
        self.inner = inner

    def describe(self, idx):
        return f"video {idx[0]}, " + ", ".join(f"{name} {i}" for name, i in zip(self.inner, idx[1:]))


def check_bound(got, ref, bound, layout):
    """Assert |got - ref| <= bound element by element (NaN fails); on failure report the worst element in kernel terms."""
    got = got.to(device=ref.device, dtype=torch.float64)
    ref = ref.to(torch.float64)
    bound = torch.as_tensor(bound, dtype=torch.float64, device=ref.device).expand_as(ref)
    err = (got - ref).abs()
    bad = ~(err <= bound)
    if not bool(bad.any()):
        return
    ratio = torch.where(bad, err / bound.clamp_min(1e-300), torch.zeros_like(err))
    ratio = torch.where(torch.isnan(ratio), torch.full_like(ratio, math.inf), ratio)
    idx = tuple(int(i) for i in torch.unravel_index(torch.argmax(ratio), ratio.shape))
    raise AssertionError(
        f"{int(bad.sum())} of {ref.numel()} elements out of bound; worst at {layout.describe(idx)}: got {float(got[idx]):.9g}, "
        f"reference {float(ref[idx]):.9g}, |error| {float(err[idx]):.3g} > bound {float(bound[idx]):.3g}")


def gemm_reference(As, Ws, scale, bias_mix, rows_per_video):
    """fp64 (ref, mag) of out[m] = sum_s scale[v, s] (A_s W_s^T)[m] + bias_mix[v], v = m // rows_per_video, from the kernel's inputs."""
    M, N = As[0].shape[0], Ws[0].shape[0]
    srow = scale.double().repeat_interleave(rows_per_video, 0)
    ref = torch.zeros((M, N), dtype=torch.float64, device=As[0].device)
    mag = torch.zeros_like(ref)
    for s, (a, w) in enumerate(zip(As, Ws)):
        a, w = a.double(), w.double()
        ref += srow[:, s:s + 1] * (a @ w.T)
        mag += srow[:, s:s + 1].abs() * (a.abs() @ w.abs().T)
    if bias_mix is not None:
        b = bias_mix.double().repeat_interleave(rows_per_video, 0)
        ref += b
        mag += b.abs()
    return ref, mag


def gemm_bound(ref, mag, Ks):
    return BF16_REL * ref.abs() + 4 * U * (sum(Ks) + len(Ks)) * mag


def _scale_rows(B, nseg):
    """Distinct mixing-weight rows: neighbouring videos differ by at least 0.2 in every segment, and no two rows are equal."""
    v = torch.arange(B, dtype=torch.float64)[:, None]
    s = torch.arange(nseg, dtype=torch.float64)[None, :]
    return (0.2 + 0.1 * torch.remainder(5 * v + 3 * s, 7) + 0.0005 * v).float()


def make_gemm_case(B, rows_per_video, Ks, N, seed, bias=True, device="cpu"):
    """Operands with a positive mean, so that |ref| is of the order of mag and the per-element bound is tight everywhere."""
    g = torch.Generator().manual_seed(seed)
    M = B * rows_per_video
    As = [torch.rand(M, k, generator=g).to(torch.bfloat16) for k in Ks]
    Ws = [((torch.rand(N, k, generator=g) - 0.3) / math.sqrt(k)).to(torch.bfloat16) for k in Ks]
    scale = _scale_rows(B, len(Ks))
    bias_mix = torch.randn(B, N, generator=g) * 0.5 + 0.25 if bias else None
    mv = lambda t: None if t is None else t.to(device)  # noqa: E731
    return [mv(a) for a in As], [mv(w) for w in Ws], mv(scale), mv(bias_mix)


# ---- the harness catches what it must (CPU) --------------------------------------------------------------------------------------------
SELF_B, SELF_RPV, SELF_KS, SELF_N = 10, 27, (200, 8, 136, 72), 136


@pytest.fixture(scope="module")
def self_case():
    As, Ws, scale, bias_mix = make_gemm_case(SELF_B, SELF_RPV, SELF_KS, SELF_N, seed=11)
    ref, mag = gemm_reference(As, Ws, scale, bias_mix, SELF_RPV)
    return As, Ws, scale, bias_mix, ref, gemm_bound(ref, mag, SELF_KS)


def _rounded(ref):
    return ref.to(torch.bfloat16)


def test_bound_passes_the_rounded_reference(self_case):
    *_, ref, bound = self_case
    check_bound(_rounded(ref), ref, bound, GemmLayout(SELF_RPV))


def _mutated(self_case, kind):
    As, Ws, scale, bias_mix, ref, _ = self_case
    if kind == "three_ulps":
        got = _rounded(ref).float()
        # the element where the bound is tightest relative to its value: the harness must resolve 3 bf16 ulps there
        idx = int(torch.argmax(ref.abs() / self_case[-1]))
        m, n = divmod(idx, SELF_N)
        x = float(got[m, n])
        got[m, n] = x + 3 * 2.0 ** (math.floor(math.log2(abs(x))) - 7)
        return got
    if kind == "swapped_scales":  # videos 2 and 3 both lie in rows 54..107 of the first 128-row tile
        sc = scale.clone()
        assert (sc[2] - sc[3]).abs().min() >= 0.1
        sc[[2, 3]] = sc[[3, 2]]
        return _rounded(gemm_reference(As, Ws, sc, bias_mix, SELF_RPV)[0])
    if kind == "dropped_k_tail":  # the last 8 columns of segment 0 (K = 200: the tail of its fourth k-block)
        a0 = As[0].clone()
        a0[:, -8:] = 0
        return _rounded(gemm_reference([a0, *As[1:]], Ws, scale, bias_mix, SELF_RPV)[0])
    if kind == "neighbour_bias_row":
        bm = bias_mix.clone()
        bm[4] = bm[5]
        return _rounded(gemm_reference(As, Ws, scale, bm, SELF_RPV)[0])
    if kind == "zero_box":  # one 128-row x 32-column output box never stored
        got = _rounded(ref).clone()
        got[TILE_M:2 * TILE_M, BOX_N:2 * BOX_N] = 0
        return got
    raise ValueError(kind)


@pytest.mark.parametrize("kind,where", [("three_ulps", ("column",)), ("swapped_scales", ("video 2,", "video 3,")), ("dropped_k_tail", ("video",)),
                                        ("neighbour_bias_row", ("video 4,",)), ("zero_box", ("row block 1, column block 0), 32-column output box 1",))])
def test_bound_fails_on_each_mutation(self_case, kind, where):
    """The failure message names where the mistake is, in the terms a tiling change would be debugged in."""
    *_, ref, bound = self_case
    with pytest.raises(AssertionError, match="out of bound") as e:
        check_bound(_mutated(self_case, kind), ref, bound, GemmLayout(SELF_RPV))
    assert any(w in str(e.value) for w in where), str(e.value)


def test_weights_bound_fails_on_swapped_neighbour_weights():
    """Two videos with close weights: swapping their weight rows is still caught by the relative weights bound."""
    s = torch.tensor([[0.0, 1.0, 2.0], [0.0, 1.0, 2.0001]], dtype=torch.float32)
    w64 = torch.softmax(s.double(), -1)
    got = w64.float()[[1, 0]]
    check_bound(w64.float(), w64, weights_bound(s, w64), VideoLayout())
    with pytest.raises(AssertionError, match="video"):
        check_bound(got, w64, weights_bound(s, w64), VideoLayout())


# ---- scores, softmax and mix: references and bounds -------------------------------------------------------------------------------------
def weights_bound(scores, w64):
    s = scores.double()
    return (16 + (s - s.max(-1, keepdim=True).values).abs()) * U * w64 + TINY


def check_weights(w, scores, layout=None):
    """w (fp32 [B, E]) against the fp64 softmax of the fp32 scores, its row sums, and the exact E = 1 case."""
    layout = layout or VideoLayout()
    w64 = torch.softmax(scores.double(), -1)
    assert not torch.isnan(w).any()
    check_bound(w, w64, weights_bound(scores, w64), layout)
    E = w.shape[1]
    check_bound(w.double().sum(-1, keepdim=True), torch.ones_like(w64[:, :1]), E * U * (1 + 1e-6), VideoLayout(("sum over segments",)))
    if E == 1:
        assert torch.equal(w, torch.ones_like(w))


def _stream():
    return torch.cuda.current_stream().cuda_stream


COUNTS = (1, 37, 256, 257, 4096)


def _partials(B, E, seed):
    g = torch.Generator().manual_seed(seed)
    counts = [COUNTS[(e + seed) % len(COUNTS)] for e in range(E)]
    parts = [(torch.randn(B, n, generator=g) + 0.3 * (e - 1)).to(DEV) for e, n in enumerate(counts)]
    consts = [None if e % 3 == 1 else torch.tensor([0.5 * e - 1.0], device=DEV) for e in range(E)]
    return parts, counts, consts


def scores_reference(parts, consts, T):
    """(ref, bound) [B, E] of s = (1/T) sum_i p_i + c."""
    ref, bound = [], []
    for p, c in zip(parts, consts):
        p = p.double()
        c = 0.0 if c is None else float(c)
        ref.append(p.sum(-1) / T + c)
        bound.append((math.ceil(p.shape[1] / 256) + 12) * U * (p.abs().sum(-1) / T + abs(c)))
    return torch.stack(ref, -1), torch.stack(bound, -1)


def _spread_scores(B, E, seed):
    """Row groups with spreads 0, 1, 30 and 200, and rows of equal scores at +1e4 and -1e4."""
    g = torch.Generator().manual_seed(seed)
    groups = []
    per = -(-B // 6)
    for spread in (0.0, 1.0, 30.0, 200.0):
        r = torch.rand(per, E, generator=g, dtype=torch.float64)
        if E >= 2:
            r[:, 0], r[:, -1] = 0.0, 1.0  # the whole spread is present in every row
        groups.append(torch.randn(per, 1, generator=g, dtype=torch.float64) * 3 + spread * r)
    groups += [torch.full((per, E), 1e4, dtype=torch.float64), torch.full((per, E), -1e4, dtype=torch.float64)]
    return torch.cat(groups)[:B].float().to(DEV)


def _ptrs(ts):
    from merv_b200._lib import ptr_array

    return ptr_array([0 if t is None else t.data_ptr() for t in ts])


# ---- merv_scores_from_partials ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("E", range(1, 9))
def test_scores_from_partials_meets_bound(E):
    from merv_b200 import ops

    B, T = 300, 27
    parts, counts, consts = _partials(B, E, seed=E)
    got = ops.scores_from_partials(parts, consts, B, T)
    ref, bound = scores_reference(parts, consts, T)
    check_bound(got, ref, bound, VideoLayout())
    if E == 5:  # no constants at all: a NULL array
        got = ops.scores_from_partials(parts, None, B, T)
        ref, bound = scores_reference(parts, [None] * E, T)
        check_bound(got, ref, bound, VideoLayout())


# ---- merv_softmax_weights_ex ---------------------------------------------------------------------------------------------------------
def _biases(E, N, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    return [None if e % 3 == 2 else (torch.randn(N, generator=g) + e).to(dtype).to(DEV) for e in range(E)]


def bias_mix_reference(w, biases, N):
    """(ref, bound) [B, N] of sum_e w_e b_e from the kernel's fp32 weights; NULL biases contribute nothing."""
    E = w.shape[1]
    ref = torch.zeros((w.shape[0], N), dtype=torch.float64, device=w.device)
    mag = torch.zeros_like(ref)
    for e, b in enumerate(biases):
        if b is not None:
            ref += w[:, e:e + 1].double() * b.double()[None]
            mag += w[:, e:e + 1].double().abs() * b.double().abs()[None]
    return ref, (E + 1) * U * mag


@pytest.mark.gpu
@pytest.mark.parametrize("bias_dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("N", [8, 264, 4104])
@pytest.mark.parametrize("E", [1, 2, 5, 8])
def test_softmax_weights_ex_meets_bounds(bias_dtype, N, E):
    from merv_b200 import _lib

    lib = _lib.load()
    B, PAD = 300, 300
    scores = _spread_scores(B, E, seed=N + E)
    biases = _biases(E, N, bias_dtype, seed=E)
    wbuf = torch.full((B * E + PAD,), -5.0, device=DEV)
    w16buf = torch.full((B * E + PAD,), -5.0, device=DEV, dtype=torch.bfloat16)
    bmbuf = torch.full((B * N + PAD,), -5.0, device=DEV)
    code = _lib.MERV_F32 if bias_dtype == torch.float32 else _lib.MERV_BF16
    _lib.check(lib.merv_softmax_weights_ex(scores.data_ptr(), wbuf.data_ptr(), w16buf.data_ptr(), _ptrs(biases), bmbuf.data_ptr(), B, E, N,
                                           code, _stream()))
    torch.cuda.synchronize()
    w, w16, bm = wbuf[:B * E].view(B, E), w16buf[:B * E].view(B, E), bmbuf[:B * N].view(B, N)
    for buf in (wbuf, w16buf, bmbuf):
        assert (buf[-PAD:] == -5.0).all(), "written past the end of an output"
    check_weights(w, scores)
    assert torch.equal(w16, w.to(torch.bfloat16))
    ref, bound = bias_mix_reference(w, biases, N)
    assert not torch.isnan(bm).any()
    check_bound(bm, ref, bound, VideoLayout(("column",)))


# ---- merv_scores_softmax_weights: one launch, bit-identical to the pair ---------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("E", range(1, 9))
def test_scores_softmax_weights_is_bit_identical_to_the_pair(E):
    from merv_b200 import _lib, ops

    lib = _lib.load()
    B, T, N = 37, 27, 264
    parts, counts, consts = _partials(B, E, seed=10 + E)
    biases = _biases(E, N, torch.bfloat16, seed=E)
    scores, w, bm = (torch.empty((B, E), device=DEV), torch.empty((B, E), device=DEV), torch.empty((B, N), device=DEV))
    w16 = torch.empty((B, E), device=DEV, dtype=torch.bfloat16)
    _lib.check(lib.merv_scores_softmax_weights(_ptrs(parts), _lib.i32_array(counts), _ptrs(consts), _ptrs(biases), scores.data_ptr(),
                                               w.data_ptr(), w16.data_ptr(), bm.data_ptr(), B, E, T, N, _stream()))
    want_s = ops.scores_from_partials(parts, consts, B, T)
    want_w, want_bm = torch.empty((B, E), device=DEV), torch.empty((B, N), device=DEV)
    want_w16 = torch.empty((B, E), device=DEV, dtype=torch.bfloat16)
    _lib.check(lib.merv_softmax_weights_ex(want_s.data_ptr(), want_w.data_ptr(), want_w16.data_ptr(), _ptrs(biases), want_bm.data_ptr(), B, E,
                                           N, _lib.MERV_BF16, _stream()))
    torch.cuda.synchronize()
    assert torch.equal(scores, want_s) and torch.equal(w, want_w) and torch.equal(w16, want_w16) and torch.equal(bm, want_bm)
    ref, bound = scores_reference(parts, consts, T)
    check_bound(scores, ref, bound, VideoLayout())
    check_weights(w, scores)


# ---- merv_softmax_mix --------------------------------------------------------------------------------------------------------------
def mix_reference(Vs, w, T, dtype):
    """(ref, bound) [B, T, K] of sum_e w_e V_e with the kernel's weights; single-token encoders are broadcast over the T tokens."""
    E = len(Vs)
    ref = torch.zeros((Vs[0].shape[0], T, Vs[0].shape[2]), dtype=torch.float64, device=Vs[0].device)
    mag = torch.zeros_like(ref)
    for e, v in enumerate(Vs):
        we = w[:, e].double()[:, None, None]
        ref += we * v.double()
        mag += we.abs() * v.double().abs()
    bound = (E + 1) * U * mag
    if dtype == torch.bfloat16:
        bound = bound + BF16_REL * ref.abs()
    return ref, bound


def _mix_inputs(B, T, K, E, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    single = E // 2 if E >= 2 else None  # one single-token encoder among the others
    Vs = [(torch.randn(B, 1 if e == single else T, K, generator=g) + 0.5 * e).to(dtype).to(DEV) for e in range(E)]
    return Vs, _spread_scores(B, E, seed)[:, :E].contiguous()


def _check_mix(Vs, T, scores, dtype):
    from merv_b200 import ops

    out, w = ops.softmax_mix(Vs, T, scores=scores)
    out2, w2 = ops.softmax_mix(Vs, T, weights=w.clone())
    torch.cuda.synchronize()
    assert torch.equal(out, out2), "scores= and weights= modes differ for the same weights"
    check_weights(w, scores)
    ref, bound = mix_reference(Vs, w, T, dtype)
    check_bound(out, ref, bound, VideoLayout(("token", "column")))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("E", range(1, 9))
@pytest.mark.parametrize("K", ["min", 200, 4096])
def test_softmax_mix_meets_bound(dtype, E, K):
    if K == "min":
        K = 8 if dtype == torch.bfloat16 else 4
    B, T = 6, 27
    Vs, scores = _mix_inputs(B, T, K, E, dtype, seed=E * 7 + K)
    _check_mix(Vs, T, scores, dtype)


def _mix_grid(B, T, K, vec, sms):
    """(CTAs per video, vectors per video) as merv_softmax_mix chooses them (mix.cu: launch_mix)."""
    nvec = T * (K // vec)
    return min(-(-nvec // 512), max(sms * 64 // B, 1)), nvec


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,K", [(torch.float32, 1024), (torch.bfloat16, 2040)])
def test_softmax_mix_grid_stride_loop(dtype, K):
    """B = 300, T = 64: few CTAs per video, so each thread runs the grid-stride loop more than once and its last pass has no second vector."""
    from merv_b200 import ops

    B, T, E = 300, 64, 4
    gx, nvec = _mix_grid(B, T, K, 8 if dtype == torch.bfloat16 else 4, ops.num_sms())
    stride = gx * 256
    assert 2 * stride < nvec and 0 < nvec % (2 * stride) <= stride, "shape no longer exercises the loop and its tail on this GPU"
    Vs, scores = _mix_inputs(B, T, K, E, dtype, seed=3)
    _check_mix(Vs, T, scores, dtype)


# ---- merv_fused_linear_mix ------------------------------------------------------------------------------------------------------------
# name: (videos, rows_per_video, per-segment K, N, bias_mix)
GEMM_CASES = {
    "merv_full": (2, 1024, (1024, 1024, 768, 768), 4096, True),
    "ragged4_n136_r27": (11, 27, (200, 8, 136, 72), 136, True),
    "ragged3_n264_r96": (5, 96, (200, 8, 136), 264, True),
    "ragged2_n8_r1": (300, 1, (136, 72), 8, True),
    "k64_n4096_r128_nobias": (3, 128, (64,), 4096, False),
    "k64_n264_r64": (7, 64, (64,), 264, True),
    "full_k_n4104_r27": (9, 27, (1024, 1024, 768, 768), 4104, True),
}
_GEMM_REFS = {}


def _gemm_case(name):
    if name not in _GEMM_REFS:
        B, rpv, Ks, N, bias = GEMM_CASES[name]
        As, Ws, scale, bias_mix = make_gemm_case(B, rpv, Ks, N, seed=sum(map(ord, name)), bias=bias, device=DEV)
        ref, mag = gemm_reference(As, Ws, scale, bias_mix, rpv)
        _GEMM_REFS.clear()  # one case at a time on the device
        _GEMM_REFS[name] = (As, Ws, scale, bias_mix, ref, gemm_bound(ref, mag, Ks))
    return _GEMM_REFS[name]


def _run_gemm(name, monkeypatch, cta_group, wide, **kw):
    from merv_b200 import ops

    monkeypatch.setenv("MERV_GEMM_CTA_GROUP", str(cta_group))
    monkeypatch.setenv("MERV_GEMM_WIDE_OUT", str(wide))
    As, Ws, scale, bias_mix, _, _ = _gemm_case(name)
    out = ops.fused_linear_mix(As, Ws, scale, bias_mix, GEMM_CASES[name][1], **kw)
    torch.cuda.synchronize()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("cta_group", [1, 2])
@pytest.mark.parametrize("name", list(GEMM_CASES))
def test_fused_linear_mix_meets_bound(name, cta_group, monkeypatch):
    """Both epilogue stagings meet the bound and are bit-identical: only the shape of the staged output box differs."""
    *_, ref, bound = _gemm_case(name)
    layout = GemmLayout(GEMM_CASES[name][1])
    narrow = _run_gemm(name, monkeypatch, cta_group, 0)
    check_bound(narrow, ref, bound, layout)
    wide = _run_gemm(name, monkeypatch, cta_group, 1)
    check_bound(wide, ref, bound, layout)
    assert torch.equal(narrow, wide), "MERV_GEMM_WIDE_OUT changed the arithmetic"


@pytest.mark.gpu
@pytest.mark.parametrize("cta_group", [1, 2])
@pytest.mark.parametrize("name", ["merv_full", "ragged4_n136_r27", "k64_n264_r64"])
def test_fused_linear_mix_capped_grid_is_bit_identical(name, cta_group, monkeypatch):
    """max_ctas caps the persistent grid: every tile does the same arithmetic whichever CTA (pair) takes it."""
    want = _run_gemm(name, monkeypatch, cta_group, 0, max_ctas=0)
    for max_ctas in (1, 2, 3, 7):
        got = _run_gemm(name, monkeypatch, cta_group, 0, max_ctas=max_ctas)
        assert torch.equal(got, want), f"max_ctas={max_ctas} differs from the full grid"


SENTINEL = 0x7FA5  # a NaN payload: bitwise comparisons only


def _sentinel(shape):
    return torch.full(shape, SENTINEL, dtype=torch.int16, device=DEV).view(torch.bfloat16)


@pytest.mark.gpu
@pytest.mark.parametrize("cta_group,wide", [(1, 0), (2, 0), (2, 1)])
@pytest.mark.parametrize("name", ["ragged4_n136_r27", "k64_n4096_r128_nobias", "ragged2_n8_r1"])
def test_fused_linear_mix_writes_only_its_block(name, cta_group, wide, monkeypatch):
    """A wider preallocated output (ldo > N) at a row and column offset: the block is the flat result, nothing around it is touched."""
    B, rpv, _, N, _ = GEMM_CASES[name]
    M = B * rpv
    flat = _run_gemm(name, monkeypatch, cta_group, wide)
    buf = _sentinel((M + 130, N + 64))
    out = _run_gemm(name, monkeypatch, cta_group, wide, out=buf[65:65 + M, 16:16 + N])
    assert out.data_ptr() == buf[65:, 16:].data_ptr()
    assert torch.equal(buf[65:65 + M, 16:16 + N], flat)
    outside = torch.ones(buf.shape, dtype=torch.bool, device=DEV)
    outside[65:65 + M, 16:16 + N] = False
    assert (buf.view(torch.int16)[outside] == SENTINEL).all(), "the GEMM wrote outside its [M, N] block"


@pytest.mark.gpu
@pytest.mark.parametrize("cta_group,wide", [(1, 0), (2, 0), (2, 1)])
def test_fused_linear_mix_batch_strided_slot(cta_group, wide, monkeypatch):
    """[B, rows_per_video + 9, N] buffer, prefix written into its [:, 3:3 + rows_per_video] slot (rows_per_video % 128 == 0)."""
    name = "k64_n4096_r128_nobias"
    B, rpv, _, N, _ = GEMM_CASES[name]
    flat = _run_gemm(name, monkeypatch, cta_group, wide)
    buf = _sentinel((B, rpv + 9, N))
    _run_gemm(name, monkeypatch, cta_group, wide, out=buf[:, 3:3 + rpv])
    assert torch.equal(buf[:, 3:3 + rpv].reshape(B * rpv, N), flat)
    rest = torch.cat([buf[:, :3], buf[:, 3 + rpv:]], 1)
    assert (rest.view(torch.int16) == SENTINEL).all(), "the GEMM wrote outside the prefix slot"


# ---- merv_fused_forward against its own three launches --------------------------------------------------------------------------------
# name: (videos, frames, patch grid side per encoder, channels per encoder, out_frames, out_size, N); merv-full has the shipped 16 x 16
# and 14 x 14 grids (the latter with overlapping windows), the 7 x 7 grid pools to 3 x 3 with overlapping windows too
FWD_CASES = {
    "merv_full": (2, 16, (16, 16, 14, 14), (1024, 1024, 768, 768), 16, 8, 4096),
    "grid7_e1": (5, 5, (7,), (136,), 3, 3, 264),
    "grid7_e3": (5, 5, (7, 7, 7), (64, 136, 200), 3, 3, 264),
}


def _fwd_inputs(name):
    B, Fr, Hs, Cs, T, S, N = FWD_CASES[name]
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    E = len(Cs)
    # a mean per (video, encoder): every video gets its own mixing weights, so a weight or bias row read for the wrong video shows
    mu = torch.remainder(torch.arange(B)[:, None] * 3 + torch.arange(E)[None, :] * 2, 5) * 0.3 - 0.6
    xs = [(torch.randn(B, Fr, h * h, c, generator=g) + mu[:, e, None, None, None]).to(torch.bfloat16).to(DEV) for e, (h, c) in enumerate(zip(Hs, Cs))]
    vs = [(torch.randn(c, generator=g) * 2 / math.sqrt(c) + 0.5 / c).to(DEV) for c in Cs]
    cs = [torch.tensor([0.3 * e], device=DEV) for e in range(E)]
    Ws = [((torch.rand(N, c, generator=g) - 0.3) / math.sqrt(c)).to(torch.bfloat16).to(DEV) for c in Cs]
    biases = [None if e == 1 else (torch.randn(N, generator=g) * 0.5).to(torch.bfloat16).to(DEV) for e in range(E)]
    return B, T, S, N, xs, vs, cs, Ws, biases


def _pool64(x, T, S):
    B, Fr, Np, C = x.shape
    H = int(math.isqrt(Np))
    y = F.adaptive_avg_pool3d(x.double().view(B, Fr, H, H, C).permute(0, 4, 1, 2, 3), (T, S, S))
    return y.permute(0, 2, 3, 4, 1).reshape(B, T * S * S, C)


def _max_window(n_in, n_out):
    return max(-(-(i + 1) * n_in // n_out) - (i * n_in) // n_out for i in range(n_out))


def _hand_run(xs, T, S, vs, cs, Ws, biases, N):
    from merv_b200 import _lib, ops

    lib = _lib.load()
    E, B = len(xs), xs[0].shape[0]
    pooled, parts = ops.pool3d(xs, [T] * E, S, score_vecs=vs)
    rpv = T * S * S
    scores, w, bm = torch.empty((B, E), device=DEV), torch.empty((B, E), device=DEV), torch.empty((B, N), device=DEV)
    w16 = torch.empty((B, E), device=DEV, dtype=torch.bfloat16)
    _lib.check(lib.merv_scores_softmax_weights(_ptrs(parts), _lib.i32_array([p.shape[1] for p in parts]), _ptrs(cs), _ptrs(biases),
                                               scores.data_ptr(), w.data_ptr(), w16.data_ptr(), bm.data_ptr(), B, E, rpv, N, _stream()))
    out = ops.fused_linear_mix(pooled, Ws, w, bm, rpv)
    torch.cuda.synchronize()
    return pooled, parts, scores, w, w16, bm, out.view(B, rpv, N)


@pytest.mark.gpu
@pytest.mark.parametrize("pdl", ["1", "0"])
@pytest.mark.parametrize("name", list(FWD_CASES))
def test_fused_forward_matches_its_three_launches(name, pdl, monkeypatch):
    from merv_b200 import ops

    monkeypatch.setenv("MERV_PDL", pdl)
    monkeypatch.delenv("MERV_POOL_ASSIST", raising=False)
    for var in ("MERV_GEMM_CTA_GROUP", "MERV_GEMM_WIDE_OUT"):
        monkeypatch.delenv(var, raising=False)
    B, T, S, N, xs, vs, cs, Ws, biases = _fwd_inputs(name)
    E, rpv = len(xs), T * S * S
    plan = ops.FusedLinearPlan(xs, [T] * E, S, vs, cs, Ws, biases, B, B)
    out, w16 = plan.run(xs, None, None)
    torch.cuda.synchronize()
    pooled, parts, scores, w, want_w16, bm, want = _hand_run(xs, T, S, vs, cs, Ws, biases, N)
    for e in range(E):
        assert torch.equal(plan.pooled[e], pooled[e]) and torch.equal(plan.partials[e], parts[e]), f"encoder {e}: pool differs"
    assert torch.equal(plan.scores, scores) and torch.equal(plan.weights, w) and torch.equal(w16, want_w16)
    assert torch.equal(plan.bias_mix, bm)
    assert torch.equal(out, want), "the prefix differs from the three-launch composition"

    # fp64 reference of the whole chain, from the bf16 inputs: pool, store as bf16 (what the pool kernel's output dtype holds), score,
    # softmax, mix.  The pooled tokens are checked against the unrounded pool first.
    pooled64 = [_pool64(x, T, S) for x in xs]
    for e, (p, p64, x) in enumerate(zip(pooled, pooled64, xs)):
        win = _max_window(x.shape[1], T) * _max_window(math.isqrt(x.shape[2]), S) ** 2
        check_bound(p, p64, BF16_REL * p64.abs() + (win + 2) * U * _pool64(x.abs(), T, S), VideoLayout(("token", "column")))
    prd = [p.to(torch.bfloat16).double() for p in pooled64]
    s64 = torch.stack([(p @ v.double()).sum(-1) / rpv + float(c) for p, v, c in zip(prd, vs, cs)], -1)
    w64 = torch.softmax(s64, -1)
    if E > 1:  # a weight row or bias row read for the wrong video would show
        assert (w64.max(-1).values - w64.min(-1).values).min() > 0.02, "degenerate softmax"
        assert (w64[1:] - w64[:-1]).abs().max(-1).values.min() > 0.02, "neighbouring videos have the same weights"
    bias_mix64 = sum(w64[:, e:e + 1] * b.double()[None] for e, b in enumerate(biases) if b is not None)
    ref, mag = gemm_reference([p.reshape(B * rpv, -1) for p in prd], Ws, w64, bias_mix64, rpv)
    check_bound(out.reshape(B * rpv, N), ref, gemm_bound(ref, mag, [x.shape[3] for x in xs]), GemmLayout(rpv))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["grid7_e3", "shipped_grid"])
def test_pool3d_capped_grid_is_bit_identical(name):
    from merv_b200 import ops

    if name == "shipped_grid":  # the TMA pool kernel at the shipped 16 x 16 -> 8 x 8 grid
        g = torch.Generator().manual_seed(3)
        xs = [torch.randn(2, 4, 256, c, generator=g).to(torch.bfloat16).to(DEV) for c in (1024, 768)]
        vs = [torch.randn(c, generator=g).to(DEV) for c in (1024, 768)]
        T, S = 4, 8
    else:
        _, T, S, _, xs, vs, _, _, _ = _fwd_inputs(name)
    want_y, want_p = ops.pool3d(xs, [T] * len(xs), S, score_vecs=vs, max_ctas=0)
    for max_ctas in (1, 5):
        y, p = ops.pool3d(xs, [T] * len(xs), S, score_vecs=vs, max_ctas=max_ctas)
        torch.cuda.synchronize()
        for e in range(len(xs)):
            assert torch.equal(y[e], want_y[e]) and torch.equal(p[e], want_p[e]), f"max_ctas={max_ctas}, encoder {e}"
