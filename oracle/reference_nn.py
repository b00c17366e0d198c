"""Plain-torch restatement of the reference's hot-path modules (``merv/util/nn_utils.py``).  TEST INFRASTRUCTURE ONLY.

The reference itself is not part of this repository (and cannot be installed offline), yet several tests compare the B200
modules against reference *modules*: same construction under a seed, ``from_reference`` adoption, fp32 autograd for the
gradients.  This file gives them those modules: the reference's class names, constructor signatures, module trees (hence
state-dict keys) and initialisation order, and a forward made of ordinary torch operators in the reference's order.  It is
pinned to the outputs the UNMODIFIED reference produced (``tests/golden/*.npz``, written by ``oracle/make_golden.py``) by
``tests/test_oracle.py::test_reference_restatement_matches_reference_golden``.

``oracle/ref_loader.load_reference_nn_utils`` returns this module unless ``MERV_REFERENCE_ROOT`` points at a reference checkout.
Nothing under ``merv_b200/`` imports it.
"""

from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn.init import xavier_uniform_
from torch.nn.parameter import Parameter


class LinearProjector(nn.Module):  # nn_utils.py:22-32
    def __init__(self, vision_dim: int, llm_dim: int, pre_proj_layernorm: bool = False) -> None:
        super().__init__()
        self.projector = nn.Linear(vision_dim, llm_dim, bias=True)
        self.layernorm = nn.LayerNorm(vision_dim) if pre_proj_layernorm else nn.Identity()

    def forward(self, img_patches: torch.Tensor) -> torch.Tensor:
        return self.projector(self.layernorm(img_patches))


class MLPProjector(nn.Module):  # nn_utils.py:35-59
    def __init__(self, vision_dim: int, llm_dim: int, mlp_type: str = "gelu-mlp", pre_proj_layernorm: bool = False) -> None:
        super().__init__()
        self.layernorm = nn.LayerNorm(vision_dim) if pre_proj_layernorm else nn.Identity()
        if mlp_type != "gelu-mlp":
            raise ValueError(f"Projector with `{mlp_type = }` is not supported!")
        self.projector = nn.Sequential(nn.Linear(vision_dim, llm_dim, bias=True), nn.GELU(), nn.Linear(llm_dim, llm_dim, bias=True))

    def forward(self, img_patches: torch.Tensor) -> torch.Tensor:
        return self.projector(self.layernorm(img_patches))


class MLPDeepProjector(nn.Module):  # nn_utils.py:62-83
    def __init__(self, vision_dim: int, llm_dim: int, mlp_type: str = "gelu-mlp", pre_proj_layernorm: bool = False) -> None:
        super().__init__()
        self.layernorm = nn.LayerNorm(vision_dim) if pre_proj_layernorm else nn.Identity()
        if mlp_type != "gelu-mlp":
            raise ValueError(f"Projector with `{mlp_type = }` is not supported!")
        self.projector = nn.Sequential(nn.Linear(vision_dim, llm_dim, bias=True), nn.GELU(), nn.Linear(llm_dim, llm_dim, bias=True), nn.GELU(),
                                       nn.Linear(llm_dim, llm_dim, bias=True))

    def forward(self, img_patches: torch.Tensor) -> torch.Tensor:
        return self.projector(self.layernorm(img_patches))


class FusedMLPProjector(nn.Module):  # nn_utils.py:86-108
    def __init__(self, fused_vision_dim: int, llm_dim: int, mlp_type: str = "fused-gelu-mlp", pre_proj_layernorm: bool = False) -> None:
        super().__init__()
        self.layernorm = nn.LayerNorm(fused_vision_dim) if pre_proj_layernorm else nn.Identity()
        self.initial_projection_dim = fused_vision_dim * 4
        if mlp_type != "fused-gelu-mlp":
            raise ValueError(f"Fused Projector with `{mlp_type = }` is not supported!")
        self.projector = nn.Sequential(nn.Linear(fused_vision_dim, self.initial_projection_dim, bias=True), nn.GELU(),
                                       nn.Linear(self.initial_projection_dim, llm_dim, bias=True), nn.GELU(), nn.Linear(llm_dim, llm_dim, bias=True))

    def forward(self, fused_img_patches: torch.Tensor) -> torch.Tensor:
        return self.projector(self.layernorm(fused_img_patches))


def get_mlp_projector(fused_vision_dim: int, llm_dim: int, mlp_type: str = "gelu-mlp") -> nn.Module:  # nn_utils.py:111-121
    if mlp_type == "linear":
        return LinearProjector(fused_vision_dim, llm_dim)
    if mlp_type == "gelu-mlp":
        return MLPProjector(fused_vision_dim, llm_dim, mlp_type)
    if mlp_type == "fused-gelu-mlp":
        return FusedMLPProjector(fused_vision_dim, llm_dim, mlp_type)
    if mlp_type == "none":
        return nn.Identity()
    raise ValueError(f"Projector with `{mlp_type = }` is not supported!")


def _grid(x: torch.Tensor) -> torch.Tensor:
    """"B F (H W) C -> B C F H W" with H = int(sqrt(N)) (nn_utils.py:323-327)."""
    B, Fr, N, C = x.shape
    H = int(math.sqrt(N))
    return x.reshape(B, Fr, H, N // H, C).permute(0, 4, 1, 2, 3)


def _tokens(y: torch.Tensor) -> torch.Tensor:
    """"B C F H W -> B (F H W) C"."""
    B, C = y.shape[:2]
    return y.permute(0, 2, 3, 4, 1).reshape(B, -1, C)


class AveragePoolingProjector(nn.Module):  # nn_utils.py:136-174: every frame pooled to output_size x output_size, then projected
    def __init__(self, fused_vision_dim: int, llm_dim: int, output_size: int, output_frames: int = 8, mlp_type: str = "gelu-mlp") -> None:
        super().__init__()
        self.output_size, self.output_frames = output_size, output_frames
        self.avg_pool = nn.AdaptiveAvgPool2d((output_size, output_size))
        self.projector = get_mlp_projector(fused_vision_dim, llm_dim, mlp_type)

    def forward(self, fused_img_patches: torch.Tensor) -> torch.Tensor:
        assert fused_img_patches.shape[1] == self.output_frames
        g = _grid(fused_img_patches)  # B C F H W
        B, C, Fr, H, W = g.shape
        pooled = self.avg_pool(g.permute(0, 2, 1, 3, 4).reshape(B * Fr, C, H, W))
        pooled = pooled.reshape(B, Fr, C, self.output_size, self.output_size).permute(0, 2, 1, 3, 4)
        return self.projector(_tokens(pooled))

    @property
    def output_token_length(self) -> int:
        return self.output_size * self.output_size

    @property
    def output_frame_length(self) -> int:
        return self.output_frames


class AveragePooling3DProjector(nn.Module):  # nn_utils.py:306-338: pool first, then project
    def __init__(self, fused_vision_dim: int, llm_dim: int, output_frames: int, output_size: int, mlp_type: str = "gelu-mlp") -> None:
        super().__init__()
        self.output_frames, self.output_size = output_frames, output_size
        self.avg_pooling = nn.AdaptiveAvgPool3d((output_frames, output_size, output_size))
        self.projector = get_mlp_projector(fused_vision_dim, llm_dim, mlp_type)

    def forward(self, fused_img_patches: torch.Tensor) -> torch.Tensor:
        return self.projector(_tokens(self.avg_pooling(_grid(fused_img_patches))))

    @property
    def output_token_length(self) -> int:
        return self.output_size * self.output_size

    @property
    def output_frame_length(self) -> int:
        return self.output_frames


class Convolutional3DProjector(nn.Module):  # nn_utils.py:341-377: Conv3d on the un-pooled grid, then the pool, then the projector
    def __init__(self, fused_vision_dim: int, llm_dim: int, output_frames: int, output_size: int, mlp_type: str = "gelu-mlp") -> None:
        super().__init__()
        self.output_frames, self.output_size = output_frames, output_size
        self.convolution_pooling = nn.Sequential(nn.Conv3d(fused_vision_dim, llm_dim, kernel_size=3, stride=1, padding=1),
                                                 nn.AdaptiveAvgPool3d((output_frames, output_size, output_size)))
        self.projector = get_mlp_projector(llm_dim, llm_dim, mlp_type)

    def forward(self, fused_img_patches: torch.Tensor) -> torch.Tensor:
        return self.projector(_tokens(self.convolution_pooling(_grid(fused_img_patches))))

    @property
    def output_token_length(self) -> int:
        return self.output_size * self.output_size

    @property
    def output_frame_length(self) -> int:
        return self.output_frames


class CrossAttention(nn.Module):  # nn_utils.py:380-412
    def __init__(self, dim, num_heads=12, qkv_bias=False, use_sdpa=True):
        super().__init__()
        self.num_heads = num_heads
        head_dim = dim // num_heads
        self.scale = head_dim**-0.5
        self.q = nn.Linear(dim, dim, bias=qkv_bias)
        self.kv = nn.Linear(dim, int(dim * 2), bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)
        self.use_sdpa = use_sdpa

    def forward(self, q: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        B, n, C = q.shape
        q = self.q(q).reshape(B, n, self.num_heads, C // self.num_heads).permute(0, 2, 1, 3)
        k, v = self.kv(x).reshape(B, x.shape[1], 2, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
        att = ((q @ k.transpose(-2, -1)) * self.scale).softmax(dim=-1)  # the attention SDPA computes, written out
        return self.proj((att @ v).transpose(1, 2).reshape(B, n, C))


class MLP(nn.Module):  # nn_utils.py:415-431
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.0):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self.drop(self.fc2(self.drop(self.act(self.fc1(x)))))


class CrossAttentionBlock(nn.Module):  # nn_utils.py:434-451
    def __init__(self, dim, num_heads, mlp_ratio=4.0, qkv_bias=False, out_dim=None, act_layer=nn.GELU, norm_layer=nn.LayerNorm):
        super().__init__()
        self.norm1 = norm_layer(dim)
        self.xattn = CrossAttention(dim, num_heads=num_heads, qkv_bias=qkv_bias)
        self.norm2 = norm_layer(dim)
        self.mlp = MLP(in_features=dim, hidden_features=int(dim * mlp_ratio), out_features=out_dim, act_layer=act_layer)

    def forward(self, q: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        q = q + self.xattn(q, self.norm1(x))
        return q + self.mlp(self.norm2(q))


class AttentivePooler(nn.Module):  # nn_utils.py:177-246
    def __init__(self, fused_vision_dim: int, llm_dim: int, num_query_tokens: int, num_heads: int = 8, output_frames: int = 8,
                 mlp_type: str = "gelu-mlp") -> None:
        super().__init__()
        self.num_query_tokens, self.output_frames = num_query_tokens, output_frames
        self.query_tokens = nn.Parameter(torch.zeros(1, num_query_tokens, fused_vision_dim))
        self.cross_attn = CrossAttentionBlock(dim=fused_vision_dim, num_heads=num_heads, qkv_bias=True)
        self.projector = get_mlp_projector(fused_vision_dim, llm_dim, mlp_type)
        nn.init.trunc_normal_(self.query_tokens, std=0.02)
        self.apply(self._init_weights)
        self.cross_attn.xattn.proj.weight.data.div_(math.sqrt(2.0))
        self.cross_attn.mlp.fc2.weight.data.div_(math.sqrt(2.0))

    @staticmethod
    def _init_weights(m):
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=0.02)
            if m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        B, Fr, N, C = x.shape
        assert Fr == self.output_frames
        x = x.reshape(B * Fr, N, C)
        q = self.cross_attn(self.query_tokens.repeat(B * Fr, 1, 1), x)
        y = self.projector(q)
        return y.reshape(B, Fr * y.shape[1], y.shape[2])

    @property
    def output_token_length(self) -> int:
        return self.num_query_tokens

    @property
    def output_frame_length(self) -> int:
        return self.output_frames


class CrossAttentionAdapterLearnableQuery(nn.Module):  # nn_utils.py:455-521
    def __init__(self, embed_dim=3072, llm_dim=4098, token_length=8, averagetoken=False, num_encoder=4, positional_embedding=False) -> None:
        super().__init__()
        self.llm_dim, self.token_length, self.averagetoken = llm_dim, token_length, averagetoken
        kdim = llm_dim if averagetoken else token_length * llm_dim
        self.attention = nn.MultiheadAttention(embed_dim=embed_dim, num_heads=1, dropout=0.0, batch_first=True, kdim=kdim, vdim=kdim)
        self.Q = Parameter(torch.empty((1, embed_dim)))
        self.num_encoder, self.positional_embedding = num_encoder, positional_embedding
        if positional_embedding:
            self.pe = Parameter(torch.empty((num_encoder, llm_dim)))
        xavier_uniform_(self.Q)
        if positional_embedding:
            xavier_uniform_(self.pe)

    def forward(self, projected_patch_embeddings):
        V = [e.repeat(1, self.token_length, 1) if e.shape[1] == 1 else e for e in projected_patch_embeddings]
        for e in V:
            assert e.shape[1] == self.token_length
        V = torch.stack(V, 1)  # [B, E, T, K]
        B, E, T, K = V.shape
        Q = self.Q.repeat(B, 1).unsqueeze(1)
        if self.averagetoken:
            key = V.mean(2)
            if self.positional_embedding:
                key = key + self.pe.unsqueeze(0)
        else:
            key = V.reshape(B, E, T * K)
        _, weights = self.attention(Q, key, key, need_weights=True)  # [B, 1, E]
        out = torch.bmm(weights, V.reshape(B, E, T * K)).reshape(B, T, K)
        return out, weights[:, 0]


class ScalarAdapter(nn.Module):  # nn_utils.py:524-537: always four scalars
    def __init__(self, num_encoder=4) -> None:
        super().__init__()
        self.scalar = nn.Parameter(torch.randn(4))

    def forward(self, projected_patch_embeddings):
        w = F.softmax(self.scalar, dim=0)
        out = (torch.stack(list(projected_patch_embeddings), 0) * w.view(-1, 1, 1, 1)).sum(0)
        return out, w.unsqueeze(0)
