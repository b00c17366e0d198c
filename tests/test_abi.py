"""CPU tests of the drop-in boundary: the C-ABI library loads without a GPU and exports exactly what
include/merv_fusion.h declares; the Python mirror keeps the reference's names, signatures, state-dict keys,
initialisation and error behaviour (SURVEY.md §8b)."""
import ctypes
import inspect
import json
import os
import re

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(REPO, "include", "merv_fusion.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(merv_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from merv_b200 import _lib

    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _header_functions()
    assert declared, "no declarations parsed from include/merv_fusion.h"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in merv_fusion.h but not exported by libmerv_fusion.so"
    assert sorted(_lib.EXPORTS) == declared, "Python binding and header disagree on the entry points"
    assert lib.merv_abi_version() == _lib.ABI_VERSION


def test_host_only_entry_points_work_without_gpu():
    from merv_b200 import _lib

    lib = _lib.load()
    descs = (_lib.PoolDesc * 2)()
    for d, (H, Cc) in zip(descs, ((16, 1024), (14, 768))):
        d.F, d.H, d.W, d.C, d.T, d.S = 16, H, H, Cc, 16, 8
    parts = _lib.i32_array([0, 0])
    assert lib.merv_pool3d_score_parts(descs, 2, _lib.MERV_BF16, parts) == 0
    assert list(parts) == [16 * 16 * 4, 16 * 12 * 4]  # T x (C / 64-channel slabs) x 4 warps per slab: shape-dependent only, never batch-dependent
    assert lib.merv_scores_from_tokens_workspace(2, 4, 1024, 4096) == 2 * 4 * 32


def test_argument_errors_are_reported_not_crashed():
    from merv_b200 import _lib

    lib = _lib.load()
    rc = lib.merv_pool3d(None, 1, 1, _lib.MERV_BF16, 0, None)
    assert rc == -6 and b"NULL" in lib.merv_last_error()
    rc = lib.merv_linear_bias_act(None, 0, None, 0, None, None, 0, 1, 1, 1, 0, 7, None, None, None)
    assert rc == -3 and b"dtype" in lib.merv_last_error()
    with pytest.raises(_lib.MervError):
        _lib.check(rc)


def test_no_cpu_fallback():
    import merv_b200 as M

    m = M.MervFusion.build([64, 48], 128, [4, 4], 16, "linear", text_embedding_dim=96).eval().requires_grad_(False)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m([torch.zeros(1, 4, 16, 64), torch.zeros(1, 4, 49, 48)])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.feature_fusion([torch.zeros(1, 64, 128), torch.zeros(1, 64, 128)])


def test_state_dict_keys_and_seeded_init_match_reference():
    # digests recorded from the UNMODIFIED reference built under torch.manual_seed(1024) (merv.py:87)
    import merv_b200 as M

    want = json.load(open(os.path.join(REPO, "tests", "golden", "ref_init_seed1024.json")))
    m = M.MervFusion.build([1024, 1024, 768, 768], 4096, [16] * 4, 64, "linear", seed=1024)
    sd = m.state_dict()
    assert sorted(sd) == sorted(want)
    for k, (shape, s, a) in want.items():
        assert list(sd[k].shape) == shape
        assert sd[k].double().sum().item() == pytest.approx(s, rel=0, abs=1e-9)
        assert sd[k].double().abs().sum().item() == pytest.approx(a, rel=1e-12)


@pytest.mark.parametrize("mlp_type,keys", [
    ("linear", ["projector.projector.weight", "projector.projector.bias"]),
    ("gelu-mlp", [f"projector.projector.{i}.{p}" for i in (0, 2) for p in ("weight", "bias")]),
    ("fused-gelu-mlp", [f"projector.projector.{i}.{p}" for i in (0, 2, 4) for p in ("weight", "bias")]),
])
def test_projector_state_dict_keys(mlp_type, keys):
    import merv_b200 as M

    p = M.AveragePooling3DProjector(32, 64, output_frames=4, output_size=2, mlp_type=mlp_type)
    assert sorted(p.state_dict()) == sorted(keys)
    assert p.output_token_length == 4 and p.output_frame_length == 4


def test_signatures_and_errors_mirror_reference():
    import merv_b200 as M

    sig = inspect.signature(M.AveragePooling3DProjector.__init__)
    assert list(sig.parameters)[1:] == ["fused_vision_dim", "llm_dim", "output_frames", "output_size", "mlp_type"]
    assert sig.parameters["mlp_type"].default == "gelu-mlp"
    sig = inspect.signature(M.CrossAttentionAdapterLearnableQuery.__init__)
    assert [(k, v.default) for k, v in list(sig.parameters.items())[1:]] == [
        ("embed_dim", 3072), ("llm_dim", 4098), ("token_length", 8), ("averagetoken", False), ("num_encoder", 4),
        ("positional_embedding", False)]
    with pytest.raises(ValueError, match="is not supported"):
        M.get_mlp_projector(8, 8, "relu-mlp")
    with pytest.raises(ValueError, match="is not supported"):
        M.MLPProjector(8, 8, "linear")
    assert isinstance(M.get_mlp_projector(8, 8, "none"), torch.nn.Identity)
    assert M.MLPProjector(8, 8).output_token_length == 1
    ff = M.CrossAttentionAdapterLearnableQuery(16, 8, 4, averagetoken=True)
    with pytest.raises(AssertionError):  # nn_utils.py:494-495
        ff([torch.zeros(1, 3, 8)])


def test_adopts_reference_modules_in_place():
    from oracle.ref_loader import load_reference_nn_utils
    import merv_b200 as M

    ref = load_reference_nn_utils()

    class FakeMerv(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.projectors = torch.nn.ModuleList(
                [ref.AveragePooling3DProjector(c, 64, output_frames=4, output_size=2, mlp_type="gelu-mlp") for c in (32, 24)])
            self.feature_fusion = ref.CrossAttentionAdapterLearnableQuery(48, 64, 16, averagetoken=True)

    v = FakeMerv()
    before = {k: t.data_ptr() for k, t in v.state_dict().items()}
    M.patch_merv(v)
    after = {k: t.data_ptr() for k, t in v.state_dict().items()}
    assert before == after, "patch_merv must keep state-dict keys and share (not copy) the parameters"
    assert isinstance(v.projectors[0], M.AveragePooling3DProjector)
    assert isinstance(v.feature_fusion, M.CrossAttentionAdapterLearnableQuery)


def test_product_never_touches_the_oracle_or_a_cpu_path():
    # The oracle is test infrastructure: nothing under merv_b200/ may import it (or the reference), and the compute
    # functions must not have a torch fallback branch for CPU tensors.
    import pathlib

    pkg = pathlib.Path(REPO) / "merv_b200"
    for path in list(pkg.glob("*.py")) + list((pkg / "csrc").glob("*.cu*")):
        text = path.read_text()
        for needle in ("import oracle", "from oracle", "/root/reference", "ref_loader", "torch_port"):
            assert needle not in text, f"{path.name} references {needle!r}"
    import ast

    tree = ast.parse((pkg / "ops.py").read_text())  # code only: docstrings cite the reference ops they replace
    called = {ast.unparse(n.func) for n in ast.walk(tree) if isinstance(n, ast.Call)}
    for needle in ("torch.matmul", "torch.mm", "torch.bmm", "F.linear", "torch.nn.functional.linear", "F.adaptive_avg_pool3d",
                   "torch.softmax", "F.softmax", "F.gelu", "torch.einsum", "torch.stack"):
        assert needle not in called, f"ops.py calls a torch compute op: {needle}"


def test_integration_md_struct_sketch_matches_the_abi():
    # the ctypes sketch a maintainer would paste from INTEGRATION.md §2 must list merv_pool_desc's fields in ABI order
    from merv_b200 import _lib

    text = open(os.path.join(REPO, "INTEGRATION.md")).read()
    block = text[text.index("class merv_pool_desc(ctypes.Structure)"):text.index("class AveragePooling3DProjector(TokenResampler)")]
    documented = re.findall(r'\("([A-Za-z_]+)",\s*ctypes\.(c_[a-z0-9_]+)\)', block)
    actual = [(name, ctype.__name__) for name, ctype in _lib.PoolDesc._fields_]
    norm = lambda t: {"c_int": "c_int32", "c_long": "c_int64", "c_longlong": "c_int64"}.get(t, t)  # noqa: E731  (ctypes aliases the fixed-width names)
    assert [(n, norm(t)) for n, t in documented] == [(n, norm(t)) for n, t in actual]
    # ... and the header declares the same order
    hdr = open(os.path.join(REPO, "include", "merv_fusion.h")).read()
    struct = hdr[hdr.index("typedef struct {"):hdr.index("} merv_pool_desc;")]
    struct = re.sub(r"/\*.*?\*/", "", struct, flags=re.S)
    names = [n for decl in struct.split(";") for n in re.findall(r"[\*\s]([A-Za-z_]+)\s*(?:,|$)", decl.strip().replace("typedef struct {", ""))]
    assert names == [n for n, _ in actual], names


_CONFIGS = [
    # (arch_specifier, feature_fusion, kwargs) as in merv/conf/models.py:28-43,100-157 and the ablations it lists
    ("no-align+3davg+linear", "cross_attention_avg_lq", {}),
    ("3davg+gelu-mlp", "cross_attention_avg_lq", {}),
    ("3davg+fused-gelu-mlp", "concat_channel", {}),
    ("3davg+frame2+linear", "concat_channel_ln", {"visual_feature_length": 32}),
    ("avg+linear", "scalar", {}),
    ("attntv+gelu-mlp", "concat", {}),
    ("3dconv+linear", "cross_attention_avg_lq", {}),
    ("3davg+linear", "query_mlp", {}),  # constructed (merv.py:211-212) although MERV.forward has no branch for it
    ("3dconv+frame2+gelu-mlp", "concat_channel", {"visual_feature_length": 32}),
    ("linear", "first", {"pre_proj_layernorm": True, "visual_feature_length": 4}),
    ("gelu-mlp", "concat_channel", {"visual_feature_length": 4}),
]


@pytest.mark.parametrize("arch,fusion,kw", _CONFIGS)
def test_from_config_builds_what_merv_init_builds(arch, fusion, kw):
    """MervFusion.from_config parses the reference's config strings (merv.py:87-227) into the same module tree with the same
    seeded initial parameters as the reference classes constructed in MERV.__init__'s order."""
    import functools

    from oracle.ref_loader import load_reference_nn_utils
    import merv_b200 as M

    ref = load_reference_nn_utils()
    dims, llm, temporal, ptl = [32, 24], 48, [4, 4], 16
    vfl = kw.get("visual_feature_length", 64)
    m = M.MervFusion.from_config(dims, llm, temporal, arch_specifier=arch, feature_fusion=fusion, projector_token_length=ptl,
                                 visual_feature_length=vfl, pre_proj_layernorm=kw.get("pre_proj_layernorm", False))
    # the reference, constructed as merv.py:87-227 does
    torch.manual_seed(dims[0])
    mlp_type = "linear" if arch.endswith("linear") else "fused-gelu-mlp" if arch.endswith("fused-gelu-mlp") else "gelu-mlp"
    parts, factor = arch.split("+"), (int(re.search(r"frame(\d+)", arch).group(1)) if "frame" in arch else 1)
    if "avg" in parts:
        P = functools.partial(ref.AveragePoolingProjector, output_size=4)
    elif "attntv" in parts:
        P = functools.partial(ref.AttentivePooler, num_query_tokens=ptl, num_heads=8)
    elif "3davg" in parts:
        P = functools.partial(ref.AveragePooling3DProjector, output_size=4)
    elif "3dconv" in parts:
        P = functools.partial(ref.Convolutional3DProjector, output_size=4)
    else:
        P = None
    if P is not None:
        projs = [P(c, llm, output_frames=t // factor, mlp_type=mlp_type) for c, t in zip(dims, temporal)]
    else:
        cls = {"linear": ref.LinearProjector, "gelu-mlp": ref.MLPProjector, "fused-gelu-mlp": ref.FusedMLPProjector}[mlp_type]
        projs = [cls(c, llm, pre_proj_layernorm=kw.get("pre_proj_layernorm", False)) for c in dims]
    if fusion == "query_mlp":
        ff = ref.MLPProjector(3072, len(dims))
    elif fusion == "cross_attention_avg_lq":
        ff = ref.CrossAttentionAdapterLearnableQuery(embed_dim=3072, llm_dim=llm, token_length=vfl, averagetoken=True)
    elif fusion == "concat_channel":
        ff = ref.LinearProjector(len(dims) * llm, llm)
    elif fusion == "concat_channel_ln":
        ff = torch.nn.Sequential(torch.nn.LayerNorm(len(dims) * llm), ref.LinearProjector(len(dims) * llm, llm))
    elif fusion == "scalar":
        ff = ref.ScalarAdapter(len(dims))
    else:
        ff = None
    want = {f"projectors.{k}": v for k, v in torch.nn.ModuleList(projs).state_dict().items()}
    if ff is not None:
        want.update({f"feature_fusion.{k}": v for k, v in ff.state_dict().items()})
    got = m.state_dict()
    assert list(got) == list(want)
    for k in want:
        assert torch.equal(got[k], want[k]), k
    assert m.arch_specifier == arch and m.feature_fusion_type == fusion
    if fusion == "query_mlp":  # merv.py:610-612
        with pytest.raises(NotImplementedError):
            m([torch.zeros(1, t, 16, c) for c, t in zip(dims, temporal)])


def test_from_config_rejects_what_merv_rejects():
    import merv_b200 as M

    with pytest.raises(ValueError, match="is not supported"):  # merv.py:105
        M.MervFusion.from_config([8], 8, [2], arch_specifier="3davg+relu", feature_fusion="first")
    with pytest.raises(AssertionError, match="square number"):  # merv.py:112
        M.MervFusion.from_config([8, 8], 8, [2, 2], arch_specifier="3davg+linear", feature_fusion="first", projector_token_length=12)
    with pytest.raises(AssertionError, match="not consistent"):  # merv.py:177-183
        M.MervFusion.from_config([8, 8], 8, [2, 4], arch_specifier="3davg+linear", feature_fusion="cross_attention_avg_lq",
                                 projector_token_length=4, visual_feature_length=8)
    with pytest.raises(NotImplementedError):  # merv.py:610-612
        M.MervFusion.from_config([8, 8], 8, [2, 2], arch_specifier="3davg+linear", feature_fusion="bogus", projector_token_length=4, visual_feature_length=8)
    # the one resampler outside the accelerated path (timm RegStage blocks): loud, never a fallback
    with pytest.raises(NotImplementedError, match="not part of the accelerated path"):
        M.MervFusion.from_config([8, 8], 8, [2, 2], arch_specifier="conv+linear", feature_fusion="first")


def test_wgrad_video_workspace_encodes_the_split_policy():
    """merv_wgrad_video_workspace (no GPU needed: a B200's 148 SMs are assumed without a device): per-(video, tile, warp) dots, plus fp32
    partial tiles only where splitting a tile's videos into ranges was measured to pay — the 96-tile encoders (C = 768) from 32 videos on
    (3 ranges); never the 128-tile ones (C = 1024), never at 16 videos (profiles/r2b_mn_pair_lab.json)."""
    from merv_b200 import _lib

    lib = _lib.load()
    os.environ.pop("MERV_WGRAD_SPLIT", None)
    os.environ.pop("MERV_GEMM_CTA_GROUP", None)

    def dots(videos, n_out, c):
        d = videos * lib.merv_wgrad_video_parts(n_out, c)
        return (d + 3) // 4 * 4

    assert lib.merv_wgrad_video_parts(4096, 1024) == 32 * 4 * 16 and lib.merv_wgrad_video_parts(4096, 768) == 32 * 3 * 16
    assert lib.merv_wgrad_video_workspace(64, 4096, 1024) == dots(64, 4096, 1024)
    assert lib.merv_wgrad_video_workspace(64, 4096, 768) == dots(64, 4096, 768) + 3 * 4096 * 768
    assert lib.merv_wgrad_video_workspace(16, 4096, 768) == dots(16, 4096, 768)
    assert lib.merv_wgrad_video_workspace(0, 4096, 768) == 0
