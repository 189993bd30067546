"""Vision Transformer on hand-written sm_100a kernels — drop-in for the reference's model API.

Mirrors the public surface of /root/reference/models/vision_transformer.py (``VisionTransformer`` 444-995,
``Block`` 109-178, ``LayerScale`` 80-106, ``global_pool_nlc`` 419-441, the ``vit_*`` entrypoints 2690-2860)
and of the timm leaf layers the reference resolves through models/_compat.py:27-172 (``Attention``,
``Mlp``, ``PatchEmbed``, ``LayerNorm``, ``DropPath``): same class names, constructor kwargs, attribute
names and state_dict keys/shapes (SURVEY Appendix B).  The arithmetic is NOT PyTorch's: every forward
and backward is a sequence of libvitk.so kernels (ops.py).  Feature combinations outside the
configs' feature set raise ``NotImplementedError`` — there is no eager fallback.
"""
from __future__ import annotations

from typing import Callable, Optional, Set, Tuple, Type, Union

import torch
import torch.nn as nn

from .. import ops
from ..store import get_store, store_for, use_store
from ._registry import register_model

__all__ = ["VisionTransformer", "Block", "Attention", "Mlp", "PatchEmbed", "LayerNorm", "LayerScale", "DropPath",
           "global_pool_nlc", "trunc_normal_"]


def trunc_normal_(tensor: torch.Tensor, mean: float = 0.0, std: float = 1.0, a: float = -2.0, b: float = 2.0):
    """timm.layers.trunc_normal_ (absolute +-2 bounds)."""
    return nn.init.trunc_normal_(tensor, mean=mean, std=std, a=a, b=b)


def _to_2tuple(v):
    return (v, v) if isinstance(v, int) else tuple(v)


# --------------------------------------------------------------------------------------------------
# leaf layers
# --------------------------------------------------------------------------------------------------
class LayerNorm(nn.LayerNorm):
    """timm LayerNorm (eps=1e-6).  Stand-alone forward: fp32 in -> fp32 out on the vitk LN kernel."""

    def __init__(self, num_channels: int, eps: float = 1e-6, affine: bool = True, **kwargs):
        if not affine:
            raise NotImplementedError("LayerNorm(affine=False) is not built")
        super().__init__(num_channels, eps=eps, elementwise_affine=True)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        st = store_for(self)
        st.sync_shadow()
        st.attach_grads()
        return ops.LayerNormFn.apply(x, st.anchor, self, st, torch.is_grad_enabled())


class DropPath(nn.Module):
    """Stochastic depth per sample.  Inside ``Block`` the scale is folded into the GEMM epilogue; this
    module only carries ``drop_prob`` (and works stand-alone through a broadcast multiply)."""

    def __init__(self, drop_prob: float = 0.0, scale_by_keep: bool = True):
        super().__init__()
        if not scale_by_keep:
            raise NotImplementedError("DropPath(scale_by_keep=False) is not built")
        self.drop_prob = drop_prob
        self.scale_by_keep = scale_by_keep

    def forward(self, x):
        rs = ops.drop_path_scale(self.drop_prob, self.training, x.shape[0], x.device)
        if rs is None:
            return x
        return x * rs.view((x.shape[0],) + (1,) * (x.ndim - 1))

    def extra_repr(self):
        return f"drop_prob={round(self.drop_prob, 3):0.3f}"


class LayerScale(nn.Module):
    """/root/reference/models/vision_transformer.py:80-106."""

    def __init__(self, dim: int, init_values: float = 1e-5, inplace: bool = False):
        super().__init__()
        self.inplace = inplace
        self.gamma = nn.Parameter(init_values * torch.ones(dim))

    def forward(self, x):
        return x.mul_(self.gamma) if self.inplace else x * self.gamma


class PatchEmbed(nn.Module):
    """2D image to patch embedding: Conv2d(k = s = patch) expressed as patchify + tcgen05 GEMM."""

    def __init__(self, img_size=224, patch_size=16, in_chans=3, embed_dim=768, norm_layer=None, flatten=True,
                 output_fmt=None, bias=True, strict_img_size=True, dynamic_img_pad=False):
        super().__init__()
        if norm_layer is not None or not flatten or output_fmt is not None or dynamic_img_pad or not strict_img_size:
            raise NotImplementedError("PatchEmbed: norm_layer / output_fmt / dynamic padding are not built")
        self.patch_size = _to_2tuple(patch_size)
        self.img_size = _to_2tuple(img_size)
        if self.patch_size[0] != self.patch_size[1] or self.patch_size[0] % 8 != 0:
            raise NotImplementedError(f"PatchEmbed: patch size {self.patch_size} (square, multiple of 8 only)")
        self.grid_size = (self.img_size[0] // self.patch_size[0], self.img_size[1] // self.patch_size[1])
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.flatten = flatten
        self.strict_img_size = strict_img_size
        self.dynamic_img_pad = dynamic_img_pad
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=self.patch_size, stride=self.patch_size, bias=bias)
        self.norm = nn.Identity()

    def _check(self, x):
        B, C, H, W = x.shape
        if H != self.img_size[0] or W != self.img_size[1]:
            raise AssertionError(f"Input size ({H}*{W}) doesn't match model ({self.img_size[0]}*{self.img_size[1]}).")

    def forward(self, x):
        self._check(x)
        st = store_for(self)
        st.sync_shadow()
        st.attach_grads()
        return ops.PatchEmbedFn.apply(x, st.anchor, self, st, torch.is_grad_enabled())


class Attention(nn.Module):
    """timm Attention: qkv Linear -> SDPA (softmax dropout = attn_drop) -> proj Linear -> proj_drop (qk_norm / masks not built)."""

    fused_attn = True

    def __init__(self, dim: int, num_heads: int = 8, qkv_bias: bool = False, qk_norm: bool = False,
                 scale_norm: bool = False, proj_bias: bool = True, attn_drop: float = 0.0, proj_drop: float = 0.0,
                 norm_layer: Optional[Type[nn.Module]] = None):
        super().__init__()
        assert dim % num_heads == 0, "dim should be divisible by num_heads"
        if qk_norm or scale_norm:
            raise NotImplementedError("Attention: qk_norm / scale_norm are not built")
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        if self.head_dim % 8 != 0 or not 16 <= self.head_dim <= 80:
            raise NotImplementedError(f"Attention: head_dim={self.head_dim}; the sm_100a attention kernels run on 64-wide head "
                                      "tiles (head_dim a multiple of 8 in [16, 80]: narrower heads are zero-padded by TMA and run "
                                      "sequences of up to 4224 tokens, heads of 72 / 80 take a second tile and sequences of at most "
                                      "256 tokens)")
        self.scale = self.head_dim ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.q_norm = nn.Identity()
        self.k_norm = nn.Identity()
        self.attn_drop = nn.Dropout(attn_drop)
        self.norm = nn.Identity()
        self.proj = nn.Linear(dim, dim, bias=proj_bias)
        self.proj_drop = nn.Dropout(proj_drop)

    def forward(self, x: torch.Tensor, attn_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if attn_mask is not None:
            raise NotImplementedError("Attention: attn_mask is not built")
        st = store_for(self)
        st.sync_shadow()
        st.attach_grads()
        x = ops.AttentionFn.apply(x, st.anchor, self, st, torch.is_grad_enabled(), self.attn_drop.p if self.training else 0.0)
        if self.training and self.proj_drop.p > 0.0:   # stand-alone use; inside a Block the mask rides in the proj epilogue
            x = ops.DropoutFn.apply(x, st, "attn.proj_drop", self.proj_drop.p)
        return x


class Mlp(nn.Module):
    """timm Mlp: fc1 -> GELU(erf) -> fc2, GELU fused into the fc1 GEMM epilogue."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, norm_layer=None,
                 bias=True, drop=0.0, use_conv=False):
        super().__init__()
        if act_layer is not nn.GELU or norm_layer is not None or use_conv:
            raise NotImplementedError("Mlp: only act_layer=nn.GELU without norm/conv is built")
        drop_probs = (drop, drop) if isinstance(drop, (int, float)) else tuple(drop)
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features, bias=bias)
        self.act = nn.GELU()
        self.drop1 = nn.Dropout(drop_probs[0])
        self.norm = nn.Identity()
        self.fc2 = nn.Linear(hidden_features, out_features, bias=bias)
        self.drop2 = nn.Dropout(drop_probs[1])

    def forward(self, x):
        st = store_for(self)
        st.sync_shadow()
        st.attach_grads()
        # stand-alone use (inside a Block both masks ride in the GEMM epilogues): drop1 in the fc1 GELU epilogue, drop2 after
        x = ops.MlpFn.apply(x, st.anchor, self, st, torch.is_grad_enabled(), self.drop1.p if self.training else 0.0)
        if self.training and self.drop2.p > 0.0:
            x = ops.DropoutFn.apply(x, st, "mlp.drop2", self.drop2.p)
        return x


# --------------------------------------------------------------------------------------------------
# Block
# --------------------------------------------------------------------------------------------------
class Block(nn.Module):
    """Pre-norm transformer block (/root/reference/models/vision_transformer.py:109-178):
    ``x = x + dp1(ls1(attn(norm1 x))); x = x + dp2(ls2(mlp(norm2 x)))`` as one fused stage."""

    def __init__(self, dim: int, num_heads: int, mlp_ratio: float = 4.0, qkv_bias: bool = False, qk_norm: bool = False,
                 scale_attn_norm: bool = False, scale_mlp_norm: bool = False, proj_bias: bool = True,
                 proj_drop: float = 0.0, attn_drop: float = 0.0, init_values: Optional[float] = None,
                 drop_path: float = 0.0, act_layer: Type[nn.Module] = nn.GELU, norm_layer: Type[nn.Module] = LayerNorm,
                 mlp_layer: Type[nn.Module] = Mlp) -> None:
        super().__init__()
        if norm_layer is not LayerNorm or mlp_layer is not Mlp:
            raise NotImplementedError("Block: only norm_layer=LayerNorm and mlp_layer=Mlp are built")
        if scale_mlp_norm:
            raise NotImplementedError("Block: scale_mlp_norm is not built")
        self.norm1 = norm_layer(dim)
        self.attn = Attention(dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_norm=qk_norm, scale_norm=scale_attn_norm,
                              proj_bias=proj_bias, attn_drop=attn_drop, proj_drop=proj_drop, norm_layer=norm_layer)
        self.ls1 = LayerScale(dim, init_values=init_values) if init_values else nn.Identity()
        self.drop_path1 = DropPath(drop_path) if drop_path > 0.0 else nn.Identity()
        self.norm2 = norm_layer(dim)
        self.mlp = mlp_layer(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, bias=proj_bias,
                             drop=proj_drop)
        self.ls2 = LayerScale(dim, init_values=init_values) if init_values else nn.Identity()
        self.drop_path2 = DropPath(drop_path) if drop_path > 0.0 else nn.Identity()
        self._vitk_tag = "block"
        self._vitk_index = 0

    def _drop_probs(self):
        return (self.drop_path1.drop_prob if isinstance(self.drop_path1, DropPath) else 0.0,
                self.drop_path2.drop_prob if isinstance(self.drop_path2, DropPath) else 0.0)

    def forward(self, x: torch.Tensor, attn_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if attn_mask is not None:
            raise NotImplementedError("Block: attn_mask is not built")
        st = store_for(self)
        if st.__dict__.get("_in_root") is None:  # stand-alone use: this block is its own root
            st.sync_shadow()
            st.attach_grads()
            st.__dict__["_last_rs"] = None
        dp1, dp2 = self._drop_probs()
        masks = st.__dict__.get("_dp_masks") if st.__dict__.get("_in_root") is not None else None
        if masks is not None:      # drawn once per forward by the root model: rows 2i, 2i+1 belong to block i
            i = self._vitk_index
            rs1 = masks[2 * i] if dp1 > 0.0 else None
            rs2 = masks[2 * i + 1] if dp2 > 0.0 else None
        else:
            own = ops.drop_path_masks([dp1, dp2], x.shape[0], x.device) if self.training else None
            rs1 = own[0] if own is not None and dp1 > 0.0 else None
            rs2 = own[1] if own is not None and dp2 > 0.0 else None
        prev_rs = st.__dict__.get("_last_rs")
        # nn.Dropout sites of the block (timm Attention.proj_drop, Mlp.drop1 / drop2; one rate: Block(proj_drop=...)): three keep
        # masks per pass, applied inside the proj / fc1 / fc2 GEMM epilogues
        drop = None
        pd, pa = self.attn.proj_drop.p, self.attn.attn_drop.p
        if self.training and (pd > 0.0 or pa > 0.0):
            if self.mlp.drop1.p != pd or self.mlp.drop2.p != pd:
                raise NotImplementedError("Block: Attention.proj_drop and Mlp.drop must share one rate (Block(proj_drop=...))")
            B, N, D = x.shape
            M, F, H = B * N, self.mlp.fc1.out_features, self.attn.num_heads
            site = f"blocks.{self._vitk_index}."
            # (a site with p = 0 gets no mask; attn_drop: keep bytes [B, H, N, N] read by the attention kernels)
            drop = (ops.dropout_keep_mask(site + "attn.proj_drop", M, D, pd, x.device),
                    ops.dropout_keep_mask(site + "mlp.drop1", M, F, pd, x.device),
                    ops.dropout_keep_mask(site + "mlp.drop2", M, D, pd, x.device), 1.0 / (1.0 - pd),
                    ops.dropout_keep_mask(site + "attn.attn_drop", B * H * N, N, pa, x.device), 1.0 / (1.0 - pa))
        root = st.__dict__.get("_in_root")
        ckpt = bool(getattr(root, "grad_checkpointing", False)) and torch.is_grad_enabled()
        out = ops.BlockFn.apply(x, st.anchor, self, st, rs1, rs2, prev_rs, torch.is_grad_enabled(), self._vitk_tag, drop, ckpt)
        st.__dict__["_last_rs"] = rs2
        return out


def global_pool_nlc(x: torch.Tensor, pool_type: str = "token", num_prefix_tokens: int = 1,
                    reduce_include_prefix: bool = False):
    """/root/reference/models/vision_transformer.py:419-441 (generic helper; the model uses the fused head)."""
    if not pool_type:
        return x
    if pool_type == "token":
        return x[:, 0]
    x = x if reduce_include_prefix else x[:, num_prefix_tokens:]
    if pool_type == "avg":
        return x.mean(dim=1)
    raise NotImplementedError(f"pool type {pool_type!r} is not built ('token' and 'avg' only)")


# --------------------------------------------------------------------------------------------------
# VisionTransformer
# --------------------------------------------------------------------------------------------------
def init_weights_vit_timm(module: nn.Module, name: str = "") -> None:
    """/root/reference/models/vision_transformer.py:998-1010."""
    if isinstance(module, nn.Linear):
        trunc_normal_(module.weight, std=0.02)
        if module.bias is not None:
            nn.init.zeros_(module.bias)


class VisionTransformer(nn.Module):
    """Vision Transformer (constructor signature of /root/reference/models/vision_transformer.py:452-493)."""

    dynamic_img_size: bool = False

    def __init__(self, img_size: Union[int, Tuple[int, int]] = 224, patch_size: Union[int, Tuple[int, int]] = 16,
                 in_chans: int = 3, num_classes: int = 1000, global_pool: str = "token", embed_dim: int = 768,
                 depth: int = 12, num_heads: int = 12, mlp_ratio: float = 4.0, qkv_bias: bool = True,
                 qk_norm: bool = False, scale_attn_norm: bool = False, scale_mlp_norm: bool = False,
                 proj_bias: bool = True, init_values: Optional[float] = None, class_token: bool = True,
                 pos_embed: str = "learn", no_embed_class: bool = False, reg_tokens: int = 0, pre_norm: bool = False,
                 final_norm: bool = True, fc_norm: Optional[bool] = None, pool_include_prefix: bool = False,
                 dynamic_img_size: bool = False, dynamic_img_pad: bool = False, drop_rate: float = 0.0,
                 pos_drop_rate: float = 0.0, patch_drop_rate: float = 0.0, proj_drop_rate: float = 0.0,
                 attn_drop_rate: float = 0.0, drop_path_rate: float = 0.0, weight_init: str = "",
                 fix_init: bool = False, embed_layer: Callable = PatchEmbed, embed_norm_layer=None,
                 norm_layer=None, act_layer=None, block_fn: Type[nn.Module] = Block, mlp_layer: Type[nn.Module] = Mlp):
        super().__init__()
        assert global_pool in ("", "avg", "avgmax", "max", "token", "map")
        assert class_token or global_pool != "token"
        assert pos_embed in ("", "none", "learn")
        unsupported = dict(qk_norm=qk_norm, scale_attn_norm=scale_attn_norm, scale_mlp_norm=scale_mlp_norm,
                           no_embed_class=no_embed_class, reg_tokens=reg_tokens, pre_norm=pre_norm,
                           pool_include_prefix=pool_include_prefix, dynamic_img_size=dynamic_img_size,
                           dynamic_img_pad=dynamic_img_pad, patch_drop_rate=patch_drop_rate,
                           fix_init=fix_init, embed_norm_layer=embed_norm_layer)
        bad = {k: v for k, v in unsupported.items() if v}
        if bad:
            raise NotImplementedError(f"VisionTransformer: options outside the built fast path: {bad}")
        if global_pool not in ("avg", "token") or not class_token or pos_embed != "learn" or not final_norm:
            raise NotImplementedError("VisionTransformer: built for class_token=True, pos_embed='learn', final_norm=True, "
                                      "global_pool in ('avg', 'token')")
        if norm_layer not in (None, LayerNorm) or act_layer not in (None, nn.GELU):
            raise NotImplementedError("VisionTransformer: only LayerNorm / GELU are built")
        if embed_layer is not PatchEmbed or block_fn is not Block or mlp_layer is not Mlp:
            raise NotImplementedError("VisionTransformer: custom embed_layer / block_fn / mlp_layer are not built")
        if weight_init not in ("", "skip"):
            raise NotImplementedError(f"weight_init={weight_init!r} is not built")
        use_fc_norm = global_pool in ("avg", "avgmax", "max") if fc_norm is None else fc_norm
        if use_fc_norm != (global_pool == "avg"):
            raise NotImplementedError("fc_norm must follow the pool type (avg -> fc_norm, token -> norm)")
        norm_layer = LayerNorm
        act_layer = nn.GELU

        self.num_classes = num_classes
        self.global_pool = global_pool
        self.num_features = self.head_hidden_size = self.embed_dim = embed_dim
        self.num_prefix_tokens = 1
        self.num_reg_tokens = 0
        self.has_class_token = True
        self.no_embed_class = False
        self.pool_include_prefix = False
        self.grad_checkpointing = False

        self.patch_embed = embed_layer(img_size=img_size, patch_size=patch_size, in_chans=in_chans, embed_dim=embed_dim,
                                       bias=not pre_norm)
        num_patches = self.patch_embed.num_patches
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.reg_token = None
        embed_len = num_patches + self.num_prefix_tokens
        self.pos_embed = nn.Parameter(torch.randn(1, embed_len, embed_dim) * 0.02)
        self.pos_drop = nn.Dropout(p=pos_drop_rate)
        self.patch_drop = nn.Identity()
        self.norm_pre = nn.Identity()

        dpr = [x.item() for x in torch.linspace(0, drop_path_rate, depth, device="cpu")]  # stochastic depth decay rule
        self.blocks = nn.Sequential(*[
            block_fn(dim=embed_dim, num_heads=num_heads, mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, proj_bias=proj_bias,
                     init_values=init_values, proj_drop=proj_drop_rate, attn_drop=attn_drop_rate, drop_path=dpr[i],
                     norm_layer=norm_layer,
                     act_layer=act_layer, mlp_layer=mlp_layer)
            for i in range(depth)])
        for i, blk in enumerate(self.blocks):
            blk._vitk_tag = f"blocks.{i}."
            blk._vitk_index = i
        self.feature_info = [dict(module=f"blocks.{i}", num_chs=embed_dim, reduction=patch_size) for i in range(depth)]
        self.norm = norm_layer(embed_dim) if final_norm and not use_fc_norm else nn.Identity()
        self.attn_pool = None
        self.fc_norm = norm_layer(embed_dim) if final_norm and use_fc_norm else nn.Identity()
        self.head_drop = nn.Dropout(drop_rate)
        self.head = nn.Linear(self.embed_dim, num_classes) if num_classes > 0 else nn.Identity()
        if weight_init != "skip":
            self.init_weights(weight_init)

    # ---- init / bookkeeping (reference :634-700) ----
    def init_weights(self, mode: str = "") -> None:
        assert mode == ""
        if self.pos_embed is not None:
            trunc_normal_(self.pos_embed, std=0.02)
        if self.cls_token is not None:
            nn.init.normal_(self.cls_token, std=1e-6)
        self.apply(init_weights_vit_timm)

    def _init_weights(self, m: nn.Module) -> None:
        init_weights_vit_timm(m)

    @torch.jit.ignore
    def no_weight_decay(self) -> Set[str]:
        return {"pos_embed", "cls_token", "dist_token"}

    @torch.jit.ignore
    def group_matcher(self, coarse: bool = False):
        return dict(stem=r"^cls_token|pos_embed|patch_embed", blocks=[(r"^blocks\.(\d+)", None), (r"^norm", (99999,))])

    @torch.jit.ignore
    def set_grad_checkpointing(self, enable: bool = True) -> None:
        """/root/reference/models/vision_transformer.py:686-694, 945-946 (``checkpoint_seq`` over the blocks): every block keeps
        only its fp32 input and runs its forward kernels again at the start of its backward."""
        self.grad_checkpointing = bool(enable)

    @torch.jit.ignore
    def get_classifier(self) -> nn.Module:
        return self.head

    def reset_classifier(self, num_classes: int, global_pool: Optional[str] = None) -> None:
        self.num_classes = num_classes
        if global_pool is not None and global_pool != self.global_pool:
            raise NotImplementedError("changing global_pool after construction is not built")
        dev = self.cls_token.device
        self.head = nn.Linear(self.embed_dim, num_classes).to(dev) if num_classes > 0 else nn.Identity()
        self.__dict__.pop("_vitk_store", None)

    # ---- forward ----
    def _begin(self):
        st = get_store(self)
        st.chain.clear()
        st.sync_shadow()
        if torch.is_grad_enabled():
            st.attach_grads()
        st.__dict__["_last_rs"] = None
        return st

    def _features(self, x: torch.Tensor, st) -> torch.Tensor:
        """patch embed + tokens + pos_embed + blocks; returns the un-normalised fp32 residual stream."""
        self.patch_embed._check(x)
        if x.dtype not in (torch.float32, torch.bfloat16) or not x.is_cuda:
            raise ops.L.VitkError(f"VisionTransformer expects a float32 (or bfloat16) CUDA image batch, got {x.dtype} on {x.device}")
        if x.dtype == torch.bfloat16 and ops.PATCH_EMBED != "tma":
            x = x.float()
        x = x if x.is_contiguous() else x.contiguous()
        x = ops.EmbedFn.apply(x, st.anchor, self, st, torch.is_grad_enabled())
        if self.training and self.pos_drop.p > 0.0:   # _pos_embed ends in pos_drop (vision_transformer.py:780, deit.py:106)
            x = ops.DropoutFn.apply(x, st, "pos_drop", self.pos_drop.p)
        st.__dict__["_in_root"] = self
        # every DropPath mask of this pass in one launch, in the reference's draw order (Block.forward :175-178)
        st.__dict__["_dp_masks"] = (ops.drop_path_masks([p for blk in self.blocks for p in blk._drop_probs()],
                                                        x.shape[0], x.device) if self.training else None)
        try:
            for blk in self.blocks:
                x = blk(x)
        finally:
            st.__dict__["_in_root"] = None
            st.__dict__["_dp_masks"] = None
        return x

    def forward_features(self, x: torch.Tensor, attn_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if attn_mask is not None:
            raise NotImplementedError("attn_mask is not built")
        st = self._begin()
        with use_store(st):
            x = self._features(x, st)
            x = self.norm(x)
        return x

    def pool(self, x: torch.Tensor, pool_type: Optional[str] = None) -> torch.Tensor:
        pool_type = self.global_pool if pool_type is None else pool_type
        return global_pool_nlc(x, pool_type=pool_type, num_prefix_tokens=self.num_prefix_tokens)

    def _linear(self, lin, x, st):
        if isinstance(lin, nn.Identity):
            return x
        return ops.LinearFn.apply(x.contiguous(), st.anchor, lin, st, torch.is_grad_enabled())

    def forward_head(self, x: torch.Tensor, pre_logits: bool = False) -> torch.Tensor:
        """Generic (unfused) head on ``forward_features`` output; ``forward`` uses the fused HeadFn instead."""
        st = get_store(self)
        with use_store(st):
            x = self.pool(x).contiguous()
            x = self.fc_norm(x)
            if self.training and self.head_drop.p > 0.0:
                x = ops.DropoutFn.apply(x.contiguous(), st, "head_drop", self.head_drop.p)
            return x if pre_logits else self._linear(self.head, x, st)

    def forward(self, x: torch.Tensor, attn_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        if attn_mask is not None:
            raise NotImplementedError("attn_mask is not built")
        if isinstance(self.head, nn.Identity):
            return self.forward_head(self.forward_features(x))
        st = self._begin()
        with use_store(st):
            x = self._features(x, st)
            return ops.HeadFn.apply(x, st.anchor, self, st, st.__dict__.get("_last_rs"), torch.is_grad_enabled(),
                                    self.head_drop.p if self.training else 0.0)


# --------------------------------------------------------------------------------------------------
# entrypoints (/root/reference/models/vision_transformer.py:2690-2860; input sizes from its default_cfgs)
# --------------------------------------------------------------------------------------------------
def _create_vision_transformer(variant: str, pretrained: bool = False, **kwargs) -> VisionTransformer:
    if pretrained:
        raise NotImplementedError("pretrained weights need a network; load a state_dict instead")
    for k in ("pretrained_cfg", "pretrained_cfg_overlay", "cache_dir"):
        kwargs.pop(k, None)
    return VisionTransformer(**kwargs)


@register_model
def vit_tiny_patch16_224(pretrained: bool = False, **kwargs) -> VisionTransformer:
    """ViT-Tiny (ViT-Ti/16)"""
    model_args = dict(patch_size=16, embed_dim=192, depth=12, num_heads=3)
    return _create_vision_transformer("vit_tiny_patch16_224", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_tiny_patch16_384(pretrained: bool = False, **kwargs) -> VisionTransformer:
    model_args = dict(patch_size=16, embed_dim=192, depth=12, num_heads=3, img_size=384)
    return _create_vision_transformer("vit_tiny_patch16_384", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_small_patch16_224(pretrained: bool = False, **kwargs) -> VisionTransformer:
    """ViT-Small (ViT-S/16)"""
    model_args = dict(patch_size=16, embed_dim=384, depth=12, num_heads=6)
    return _create_vision_transformer("vit_small_patch16_224", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_small_patch16_384(pretrained: bool = False, **kwargs) -> VisionTransformer:
    model_args = dict(patch_size=16, embed_dim=384, depth=12, num_heads=6, img_size=384)
    return _create_vision_transformer("vit_small_patch16_384", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_small_patch32_224(pretrained: bool = False, **kwargs) -> VisionTransformer:
    model_args = dict(patch_size=32, embed_dim=384, depth=12, num_heads=6)
    return _create_vision_transformer("vit_small_patch32_224", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_base_patch16_224(pretrained: bool = False, **kwargs) -> VisionTransformer:
    """ViT-Base (ViT-B/16) from original paper (https://arxiv.org/abs/2010.11929)."""
    model_args = dict(patch_size=16, embed_dim=768, depth=12, num_heads=12)
    return _create_vision_transformer("vit_base_patch16_224", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_base_patch16_384(pretrained: bool = False, **kwargs) -> VisionTransformer:
    model_args = dict(patch_size=16, embed_dim=768, depth=12, num_heads=12, img_size=384)
    return _create_vision_transformer("vit_base_patch16_384", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_base_patch32_224(pretrained: bool = False, **kwargs) -> VisionTransformer:
    model_args = dict(patch_size=32, embed_dim=768, depth=12, num_heads=12)
    return _create_vision_transformer("vit_base_patch32_224", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_large_patch16_224(pretrained: bool = False, **kwargs) -> VisionTransformer:
    """ViT-Large (ViT-L/16)"""
    model_args = dict(patch_size=16, embed_dim=1024, depth=24, num_heads=16)
    return _create_vision_transformer("vit_large_patch16_224", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_large_patch16_384(pretrained: bool = False, **kwargs) -> VisionTransformer:
    """ViT-Large (ViT-L/16) at 384x384 (577 tokens): input size from the reference default_cfg (:1536-1539)."""
    model_args = dict(patch_size=16, embed_dim=1024, depth=24, num_heads=16, img_size=384)
    return _create_vision_transformer("vit_large_patch16_384", pretrained=pretrained, **dict(model_args, **kwargs))


@register_model
def vit_large_patch32_224(pretrained: bool = False, **kwargs) -> VisionTransformer:
    model_args = dict(patch_size=32, embed_dim=1024, depth=24, num_heads=16)
    return _create_vision_transformer("vit_large_patch32_224", pretrained=pretrained, **dict(model_args, **kwargs))
