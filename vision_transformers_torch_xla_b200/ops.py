"""Fused autograd stages of the ViT hot path, each a fixed sequence of libvitk.so kernel launches.

  EmbedFn  : PatchEmbed + cls/dist tokens + pos_embed          (reference vision_transformer.py:936-937)
  BlockFn  : one pre-norm transformer Block                     (reference vision_transformer.py:175-178)
  HeadFn   : pool -> (fc_)norm -> head Linear                   (reference vision_transformer.py:977-990)
  CEFn     : fused soft-target / label-smoothing / KD loss      (reference main.py:926-968)

Activations between stages are the fp32 residual stream ``[B, N, D]``; everything else is bf16 with
fp32 accumulation.  Parameter gradients are accumulated by the kernels directly into the flat fp32
gradient buffer of the ``ParamStore`` (``p.grad`` are views of it), so the autograd graph only carries
the residual-stream gradient from stage to stage.  A side channel (``store.chain``) hands the bf16,
DropPath-scaled copy of that gradient — produced for free by the LayerNorm-backward kernel — to the
next stage's backward so that no separate cast pass is needed.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib as L
from .store import ParamStore


def _empty(shape, dtype, dev):
    return torch.empty(shape, dtype=dtype, device=dev)


def _require_f32_cuda(x: torch.Tensor, what: str) -> torch.Tensor:
    if not x.is_cuda:
        raise L.VitkError(f"{what}: expected a CUDA tensor (no CPU path)")
    if x.dtype != torch.float32:
        raise L.VitkError(f"{what}: expected float32, got {x.dtype}")
    return x if x.is_contiguous() else x.contiguous()


def _bf16_grad(store: ParamStore, g: torch.Tensor, rowscale: Optional[torch.Tensor], elems_per_group: int) -> torch.Tensor:
    """bf16(rowscale * g): taken from the side channel when the producer already made it."""
    hit = store.chain.pop(g.data_ptr(), None)
    if hit is not None and hit.numel() == g.numel():
        return hit
    out = _empty(g.shape, torch.bfloat16, g.device)
    L.rowscale_cast_bf16(g, rowscale, elems_per_group, out)
    return out


# ================================================================================================
# Patch embedding + prefix tokens + positional embedding
# ================================================================================================
def _patch_grid_pad(gw: int) -> int:
    """Patch-grid width rounded up to a multiple of 8: the TMA boxes of the image operand cover 8 neighbouring patches."""
    return (gw + 7) // 8 * 8


class EmbedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, anchor, model, store: ParamStore, save: bool):
        pe = model.patch_embed
        B, C, H, W = img.shape
        ps = pe.patch_size[0]
        D = model.embed_dim
        P = pe.num_patches
        prefix = model.num_prefix_tokens
        N = P + prefix
        K = C * ps * ps
        dev = img.device
        gh, gw = pe.grid_size
        gwp = _patch_grid_pad(gw)
        x = _empty((B, N, D), torch.float32, dev)
        w = store.shadow_of(pe.proj.weight).view(D, K)
        pos = model.pos_embed.data.view(N, D)
        bias = None if pe.proj.bias is None else pe.proj.bias.data
        # 16 x 16 patches: im2col-free.  The image (cast to bf16 NCHW in one coalesced pass, or handed in as bf16 already)
        # is the GEMM's A operand through a 4-D tensor map that reads it as its patch matrix; the [B*P, C*ps*ps] matrix is
        # never materialised, neither for the forward nor for the weight gradient.  Other patch sizes: the explicit
        # im2col + cast kernel, which reads an fp32 image.
        if ps == 16 and pe.patch_size[1] == 16:
            if img.dtype == torch.bfloat16:
                src = img                         # a loader that already produces bf16 saves the cast (and half the H2D bytes)
            else:
                src = _empty(img.shape, torch.bfloat16, dev)
                L.cast_bf16(img, src)
            geom = (C, H, W, ps, gwp)
            L.gemm(src, w, x, M=B * gh * gwp, N=D, K=K, epilogue=L.EPI_PATCH, bias=bias, pos=pos, tokens_per_img=P, prefix=prefix,
                   image=("a",) + geom)
        else:
            src = _empty((B * P, K), torch.bfloat16, dev)
            L.patchify(img.float() if img.dtype == torch.bfloat16 else img, src, ps)
            geom = None
            L.gemm(src, w, x, M=B * P, N=D, K=K, epilogue=L.EPI_PATCH, bias=bias, pos=pos, tokens_per_img=P, prefix=prefix)
        xf = x.view(-1)
        posf = pos.view(-1)
        toks = [model.cls_token] + ([model.dist_token] if prefix == 2 else [])
        for j, tok in enumerate(toks):
            L.prefix_rows(xf[j * D:], tok.data.view(1, D), posf[j * D:], B, N, D, 1)
        if save:
            ctx.model, ctx.store = model, store
            ctx.src, ctx.geom = src, geom
            ctx.dims = (B, N, D, P, prefix, K)
        return x

    @staticmethod
    def backward(ctx, g):
        model, store = ctx.model, ctx.store
        B, N, D, P, prefix, K = ctx.dims
        pe = model.patch_embed
        g = _require_f32_cuda(g, "EmbedFn.backward grad")
        store.chain.pop(g.data_ptr(), None)
        dev = g.device
        toks = [model.cls_token] + ([model.dist_token] if prefix == 2 else [])
        # the token gradients are summed over the batch straight into their rows of the flat gradient buffer
        dpre = [store.grad_of(tok).view(D) if tok.requires_grad else None for tok in toks] + [None]
        dpos = store.grad_of(model.pos_embed).view(N, D) if model.pos_embed.requires_grad else None
        colsum = None if pe.proj.bias is None else store.grad_of(pe.proj.bias)
        dW = store.grad_of(pe.proj.weight).view(D, K)
        if ctx.geom is not None:
            C, H, W, ps, gwp = ctx.geom
            gh, gw = H // ps, W // ps
            rows = B * gh * gwp                    # gp in the image operand's padded row order, pad rows zeroed
            gp = _empty((rows, D), torch.bfloat16, dev)
            L.embed_bwd(g, gp, dpos, dpre[0], dpre[1], B, N, D, prefix, gw, gwp)
            L.gemm(gp, ctx.src, dW, M=D, N=K, K=rows, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, colsum=colsum,
                   image=("b",) + ctx.geom)
        else:
            gp = _empty((B * P, D), torch.bfloat16, dev)
            L.embed_bwd(g, gp, dpos, dpre[0], dpre[1], B, N, D, prefix)
            L.gemm(gp, ctx.src, dW, M=D, N=K, K=B * P, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, colsum=colsum)
        ctx.src = None
        store.fire_grad_ready()   # the last stage of every backward through the model (it takes store.anchor)
        return None, None, None, None, None


# ================================================================================================
# Transformer block
# ================================================================================================
#: test hook: callable(site, rows, cols, p, device) -> uint8 [rows, cols] keep mask (1 = keep), used INSTEAD of the Philox
#: kernel (the parity tests replay masks against the oracle; tests/test_gpu_dropout.py)
dropout_source = None
_drop_calls = 0


def dropout_keep_mask(site: str, rows: int, cols: int, p: float, device) -> Optional[torch.Tensor]:
    """Keep mask of one nn.Dropout site (timm: pos_drop, Attention.proj_drop, Mlp.drop1 / drop2, head_drop) for one forward
    pass, or None when p == 0.  Seeded like the DropPath masks: torch's CUDA seed plus a per-process call counter."""
    global _drop_calls
    if p <= 0.0:
        return None
    if not 0.0 < p < 1.0:
        raise ValueError(f"dropout probability {p} not in [0, 1)")
    if dropout_source is not None:
        m = dropout_source(site, rows, cols, p, device)
        assert m.shape == (rows, cols) and m.dtype == torch.uint8 and m.is_cuda, (site, m.shape, m.dtype)
        return m.contiguous()
    m = _empty((rows, cols), torch.uint8, device)
    _drop_calls += 1
    L.dropout_mask(m, p, torch.cuda.initial_seed() ^ 0x5DEECE66D, _drop_calls)
    return m


class DropoutFn(torch.autograd.Function):
    """nn.Dropout on an fp32 activation that has no GEMM epilogue in front of it (pos_drop; the stand-alone leaf modules)."""

    @staticmethod
    def forward(ctx, x, store, site: str, p: float):
        x = _require_f32_cuda(x, "Dropout input")
        cols = x.shape[-1]
        rows = x.numel() // cols
        mask = dropout_keep_mask(site, rows, cols, p, x.device)
        y = x.clone()
        L.mask_mul_(y, mask, 1.0 / (1.0 - p), rows, cols)
        ctx.mask, ctx.p, ctx.store = mask, p, store
        return y

    @staticmethod
    def backward(ctx, g):
        g = _require_f32_cuda(g, "Dropout grad")
        if ctx.store is not None:
            ctx.store.chain.pop(g.data_ptr(), None)   # a bf16 copy made by the consumer stage does not carry the mask
        cols = g.shape[-1]
        gx = g.clone()
        L.mask_mul_(gx, ctx.mask, 1.0 / (1.0 - ctx.p), g.numel() // cols, cols)
        ctx.mask = None
        return gx, None, None, None


class BlockFn(torch.autograd.Function):
    @staticmethod
    def _run(x, blk, store: ParamStore, rs1, rs2, drop):
        """The forward kernels of one block.  Returns (x_out, everything the backward reads)."""
        B, N, D = x.shape
        M = B * N
        H = blk.attn.num_heads
        hd = blk.attn.head_dim
        F = blk.mlp.fc1.out_features
        dev = x.device
        eps = blk.norm1.eps
        sh = store.shadow_of
        bias = lambda lin: None if lin.bias is None else lin.bias.data  # noqa: E731

        ln1 = _empty((M, D), torch.bfloat16, dev)
        mean1, rstd1 = _empty((M,), torch.float32, dev), _empty((M,), torch.float32, dev)
        L.layernorm_fwd(x, blk.norm1.weight.data, blk.norm1.bias.data, ln1, mean1, rstd1, M, D, eps)
        qkv = _empty((M, 3 * D), torch.bfloat16, dev)
        L.gemm(ln1, sh(blk.attn.qkv.weight), qkv, M=M, N=3 * D, K=D, epilogue=L.EPI_BF16, bias=bias(blk.attn.qkv))
        att = _empty((M, D), torch.bfloat16, dev)
        lse = _empty((B, H, N), torch.float32, dev)
        md1, md2, md3, dscale, ma, ascale = drop if drop is not None else (None, None, None, 1.0, None, 1.0)
        L.attn_fwd(qkv, att, lse, B, N, H, hd, blk.attn.scale, keep_mask=ma, keep_scale=ascale)
        # LayerScale (vision_transformer.py:80-106): gamma rides in the residual epilogue as a per-column scale
        g1 = blk.ls1.gamma.data if hasattr(blk.ls1, "gamma") else None
        g2 = blk.ls2.gamma.data if hasattr(blk.ls2, "gamma") else None
        x_mid = _empty((B, N, D), torch.float32, dev)
        L.gemm(att, sh(blk.attn.proj.weight), x_mid, M=M, N=D, K=D, epilogue=L.EPI_RESID, bias=bias(blk.attn.proj),
               resid=x, rowscale=rs1, rows_per_group=N, colscale=g1, mask=md1, mask_scale=dscale)
        ln2 = _empty((M, D), torch.bfloat16, dev)
        mean2, rstd2 = _empty((M,), torch.float32, dev), _empty((M,), torch.float32, dev)
        L.layernorm_fwd(x_mid, blk.norm2.weight.data, blk.norm2.bias.data, ln2, mean2, rstd2, M, D, eps)
        h = _empty((M, F), torch.bfloat16, dev)  # receives gelu'(fc1 out) (x the drop1 mask): all the backward needs of it
        act = _empty((M, F), torch.bfloat16, dev)
        L.gemm(ln2, sh(blk.mlp.fc1.weight), act, M=M, N=F, K=D, epilogue=L.EPI_GELU, bias=bias(blk.mlp.fc1), aux=h,
               mask=md2, mask_scale=dscale)
        x_out = _empty((B, N, D), torch.float32, dev)
        L.gemm(act, sh(blk.mlp.fc2.weight), x_out, M=M, N=D, K=F, epilogue=L.EPI_RESID, bias=bias(blk.mlp.fc2),
               resid=x_mid, rowscale=rs2, rows_per_group=N, colscale=g2, mask=md3, mask_scale=dscale)
        return x_out, (x, ln1, mean1, rstd1, qkv, att, lse, x_mid, ln2, mean2, rstd2, h, act)

    @staticmethod
    def forward(ctx, x, anchor, blk, store: ParamStore, rs1, rs2, prev_rs, save: bool, drop=None,
                checkpoint: bool = False):
        # drop = (keep masks of attn.proj_drop [M, D], mlp.drop1 [M, F], mlp.drop2 [M, D], 1 / (1 - p_proj),
        #         keep mask of attn.attn_drop [B * H * N, N], 1 / (1 - p_attn)) or None; a mask that is None is a site with p = 0
        # checkpoint (set_grad_checkpointing, vision_transformer.py:686-694, 945-946): keep only the block input and run the
        # forward kernels again at the start of the backward (same DropPath / dropout masks: they are inputs, not redrawn)
        x = _require_f32_cuda(x, "Block input")
        B, N, D = x.shape
        x_out, saved = BlockFn._run(x, blk, store, rs1, rs2, drop)
        if save:
            ctx.blk, ctx.store = blk, store
            ctx.dims = (B, N, D, blk.attn.num_heads, blk.attn.head_dim, blk.mlp.fc1.out_features)
            ctx.rs = (rs1, rs2, prev_rs)
            md1, _, md3, dscale, ma, ascale = drop if drop is not None else (None, None, None, 1.0, None, 1.0)
            ctx.drop = (md1, md3, dscale, ma, ascale)
            ctx.recompute = (x, drop) if checkpoint else None
            ctx.saved = None if checkpoint else saved
        return x_out

    @staticmethod
    def backward(ctx, g):
        blk, store = ctx.blk, ctx.store
        B, N, D, H, hd, F = ctx.dims
        M = B * N
        rs1, rs2, prev_rs = ctx.rs
        if ctx.recompute is not None:
            x_in, drop_in = ctx.recompute
            ctx.recompute = None
            ctx.saved = BlockFn._run(x_in, blk, store, rs1, rs2, drop_in)[1]
        x, ln1, mean1, rstd1, qkv, att, lse, x_mid, ln2, mean2, rstd2, h, act = ctx.saved
        ctx.saved = None
        g = _require_f32_cuda(g, "Block.backward grad")
        dev = g.device
        sh, gr = store.shadow_of, store.grad_of
        # weight gradient (split-K red.add into the flat grad buffer); the bias gradient (column sums of dy) rides
        # along as one extra N=16 MMA against a tile of ones inside the same kernel
        wgrad = lambda dy, xin, lin, m, n: L.gemm(  # noqa: E731
            dy, xin, gr(lin.weight), M=m, N=n, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True,
            colsum=None if lin.bias is None else gr(lin.bias))

        # ---------------- MLP branch: x_out = x_mid + rs2 * (fc2(gelu(fc1(ln2))) ) ----------------
        # LayerScale: the branch gradient is g * rs * gamma; dgamma follows from the branch's last weight gradient
        # (vitk_layerscale_grad), so the branch output never has to be stored
        def ls_bwd_scale(gb, ls):
            if hasattr(ls, "gamma"):
                L.colscale_bf16(gb, ls.gamma.data, M, D)

        def ls_bwd_grad(ls, lin):
            if hasattr(ls, "gamma") and ls.gamma.requires_grad:
                L.layerscale_grad(lin.weight.data, gr(lin.weight), None if lin.bias is None else lin.bias.data,
                                  None if lin.bias is None else gr(lin.bias), ls.gamma.data, gr(ls.gamma))

        md1, md3, dscale, ma, ascale = ctx.drop
        gb2 = _bf16_grad(store, g, rs2, N * D).view(M, D)
        ls_bwd_scale(gb2, blk.ls2)   # gb2 is exclusively ours (popped from the side channel or freshly made)
        if md3 is not None:          # Mlp.drop2 sits between fc2 and LayerScale / DropPath: its mask goes on the branch gradient
            L.mask_mul_(gb2, md3, dscale, M, D)
        wgrad(gb2, act, blk.mlp.fc2, D, F)
        ls_bwd_grad(blk.ls2, blk.mlp.fc2)
        dh = act  # reuse: gelu output is dead after the fc2 wgrad above
        # (Mlp.drop1: the saved derivative already carries mask / keep_prob, so this multiply is the same launch)
        L.gemm(gb2, sh(blk.mlp.fc2.weight), dh, M=M, N=F, K=D, epilogue=L.EPI_DGELU, b_mn=True, aux=h)
        del gb2, h
        wgrad(dh, ln2, blk.mlp.fc1, F, D)
        dln2 = ln2  # reuse: ln2 output is dead after the fc1 wgrad above
        L.gemm(dh, sh(blk.mlp.fc1.weight), dln2, M=M, N=D, K=F, epilogue=L.EPI_BF16, b_mn=True)
        del dh, act
        g_mid = _empty((B, N, D), torch.float32, dev)
        gb1 = _empty((M, D), torch.bfloat16, dev)
        L.layernorm_bwd(dln2, x_mid, mean2, rstd2, blk.norm2.weight.data, g, g_mid, gb1, rs1, N,
                        gr(blk.norm2.weight), gr(blk.norm2.bias), M, D)
        del dln2, ln2, x_mid, g

        # ---------------- attention branch: x_mid = x + rs1 * proj(attn(qkv(ln1))) ----------------
        ls_bwd_scale(gb1, blk.ls1)
        if md1 is not None:          # Attention.proj_drop
            L.mask_mul_(gb1, md1, dscale, M, D)
        wgrad(gb1, att, blk.attn.proj, D, D)
        ls_bwd_grad(blk.ls1, blk.attn.proj)
        datt = _empty((M, D), torch.bfloat16, dev)
        L.gemm(gb1, sh(blk.attn.proj.weight), datt, M=M, N=D, K=D, epilogue=L.EPI_BF16, b_mn=True)
        dqkv = _empty((M, 3 * D), torch.bfloat16, dev)
        L.attn_bwd(qkv, att, datt, lse, dqkv, B, N, H, hd, blk.attn.scale, keep_mask=ma, keep_scale=ascale)
        del gb1, datt, att, qkv, lse
        wgrad(dqkv, ln1, blk.attn.qkv, 3 * D, D)
        dln1 = ln1
        L.gemm(dqkv, sh(blk.attn.qkv.weight), dln1, M=M, N=D, K=3 * D, epilogue=L.EPI_BF16, b_mn=True)
        del dqkv
        g_in = _empty((B, N, D), torch.float32, dev)
        gb_prev = _empty((B, N, D), torch.bfloat16, dev)
        L.layernorm_bwd(dln1, x, mean1, rstd1, blk.norm1.weight.data, g_mid, g_in, gb_prev, prev_rs, N,
                        gr(blk.norm1.weight), gr(blk.norm1.bias), M, D)
        store.chain[g_in.data_ptr()] = gb_prev
        return g_in, None, None, None, None, None, None, None, None, None


# ================================================================================================
# Pool + norm + classifier head(s)
# ================================================================================================
class HeadFn(torch.autograd.Function):
    """avg:   logits = head(fc_norm(mean_{t>=prefix} x))
       token: logits = head(norm(x)[:, 0])   (+ head_dist(norm(x)[:, 1]) for the distilled model)"""

    @staticmethod
    def forward(ctx, x, anchor, model, store: ParamStore, prev_rs, save: bool, head_drop: float = 0.0):
        # head_drop > 0: nn.Dropout between fc_norm and the classifier (vision_transformer.py:987-990; the distilled
        # model's forward_head, deit.py:108-119, has none)
        x = _require_f32_cuda(x, "head input")
        B, N, D = x.shape
        dev = x.device
        prefix = model.num_prefix_tokens
        avg = model.global_pool == "avg"
        norm = model.fc_norm if avg else model.norm
        has_norm = isinstance(norm, torch.nn.LayerNorm)
        heads = [model.head] + ([model.head_dist] if getattr(model, "head_dist", None) is not None else [])
        C = heads[0].out_features
        sh = store.shadow_of
        feats, stats, outs, hmasks = [], [], [], []
        pooled = None
        if avg:
            pooled = _empty((B, D), torch.float32, dev)
            L.pool_fwd(x, pooled, B, N, D, prefix, 0)
        for j, head in enumerate(heads):
            src, ld = (pooled, D) if avg else (x.view(-1)[j * D:], N * D)
            f = _empty((B, D), torch.bfloat16, dev)
            mean, rstd = _empty((B,), torch.float32, dev), _empty((B,), torch.float32, dev)
            if has_norm:
                L.layernorm_fwd(src, norm.weight.data, norm.bias.data, f, mean, rstd, B, D, norm.eps, ld_x=ld)
            else:
                L.cast_bf16(src.view(B, -1)[:, :D].contiguous(), f)
            hmask = dropout_keep_mask("head_drop", B, D, head_drop, dev) if (head_drop > 0.0 and len(heads) == 1) else None
            if hmask is not None:
                L.mask_mul_(f, hmask, 1.0 / (1.0 - head_drop), B, D)   # the classifier and its weight gradient see the dropped features
            logits = _empty((B, C), torch.float32, dev)
            L.gemm(f, sh(head.weight), logits, M=B, N=C, K=D, epilogue=L.EPI_F32,
                   bias=None if head.bias is None else head.bias.data)
            feats.append(f)
            hmasks.append(hmask)
            stats.append((mean, rstd))
            outs.append(logits)
        if save:
            ctx.model, ctx.store = model, store
            ctx.dims = (B, N, D, C, prefix, avg, has_norm)
            ctx.saved = (x, pooled, feats, stats)
            ctx.hdrop = (hmasks, head_drop)
            ctx.prev_rs = prev_rs
        return tuple(outs) if len(outs) > 1 else outs[0]

    @staticmethod
    def backward(ctx, *dlogits):
        model, store = ctx.model, ctx.store
        B, N, D, C, prefix, avg, has_norm = ctx.dims
        x, pooled, feats, stats = ctx.saved
        ctx.saved = None
        dev = x.device
        gr, sh = store.grad_of, store.shadow_of
        norm = model.fc_norm if avg else model.norm
        heads = [model.head] + ([model.head_dist] if getattr(model, "head_dist", None) is not None else [])
        g = _empty((B, N, D), torch.float32, dev) if avg else torch.zeros((B, N, D), dtype=torch.float32, device=dev)
        for j, head in enumerate(heads):
            dl = dlogits[j]
            if dl is None:
                continue
            dl = _require_f32_cuda(dl, "dlogits")
            Cp = (C + 7) // 8 * 8  # TMA needs 16-byte row pitches: pad ragged class counts with zero columns
            if Cp != C:
                pad = torch.zeros((B, Cp), dtype=torch.float32, device=dev)
                pad[:, :C] = dl
                dl = pad
            dlb = _empty((B, Cp), torch.bfloat16, dev)
            L.cast_bf16(dl, dlb)
            L.gemm(dlb, feats[j], gr(head.weight), M=C, N=D, K=B, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True, lda=Cp,
                   colsum=None if head.bias is None else gr(head.bias))
            df = _empty((B, D), torch.bfloat16, dev)
            # K = C with row pitch Cp: both tensor maps end at the true class count, so TMA zero-fills the k >= C part
            # of the last k-block on both operands and nothing past head.weight is ever read
            L.gemm(dlb, sh(head.weight), df, M=B, N=D, K=C, epilogue=L.EPI_BF16, b_mn=True, lda=Cp)
            if ctx.hdrop[0][j] is not None:
                L.mask_mul_(df, ctx.hdrop[0][j], 1.0 / (1.0 - ctx.hdrop[1]), B, D)
            mean, rstd = stats[j]
            if not has_norm:
                raise NotImplementedError("final_norm=False head backward is not built")
            if avg:
                dpooled = _empty((B, D), torch.float32, dev)
                L.layernorm_bwd(df, pooled, mean, rstd, norm.weight.data, None, dpooled, None, None, 1,
                                gr(norm.weight), gr(norm.bias), B, D)
                L.pool_bwd(dpooled, g, B, N, D, prefix, 0)
            else:
                L.layernorm_bwd(df, x.view(-1)[j * D:], mean, rstd, norm.weight.data, None, g.view(-1)[j * D:], None,
                                None, 1, gr(norm.weight), gr(norm.bias), B, D, ld_x=N * D, ld_g=N * D)
        gb = _empty((B, N, D), torch.bfloat16, dev)
        L.rowscale_cast_bf16(g, ctx.prev_rs, N * D, gb)
        store.chain[g.data_ptr()] = gb
        return g, None, None, None, None, None, None


# ================================================================================================
# Loss
# ================================================================================================
class CEFn(torch.autograd.Function):
    """loss = (1-alpha) * CE(logits, targets) + alpha * T^2 * KL(softmax(teacher/T) || softmax(logits/T))."""

    @staticmethod
    def forward(ctx, logits, soft, labels, smoothing: float, teacher, alpha: float, temp: float):
        logits = _require_f32_cuda(logits, "loss logits")
        B, C = logits.shape
        dev = logits.device
        if soft is not None:
            soft = _require_f32_cuda(soft.to(torch.float32), "soft targets")
        if labels is not None:
            labels = labels.to(torch.int64).contiguous()
        if teacher is not None:
            teacher = _require_f32_cuda(teacher.to(torch.float32), "teacher logits")
        loss = _empty((1,), torch.float32, dev)
        dl = _empty((B, C), torch.float32, dev)
        scratch = _empty((B,), torch.float32, dev)
        L.ce_fwd_bwd(logits, soft, labels, smoothing, teacher, alpha, temp, loss, dl, scratch)
        ctx.dl = dl
        return loss.view(())

    @staticmethod
    def backward(ctx, gout):
        dl, ctx.dl = ctx.dl, None
        if dl is None:
            raise L.VitkError("the fused loss keeps one gradient buffer: backward() can run once per forward")
        gout = gout.to(torch.float32)
        L.scale_f32_(dl, gout if gout.is_contiguous() else gout.contiguous())   # upstream grad (e.g. 1/update_freq): device scalar
        return dl, None, None, None, None, None, None


#: test hook: callable(drop_probs, B, device) -> fp32 [len(drop_probs), B] of mask / keep_prob factors, used INSTEAD of
#: the Philox kernel (the parity tests replay the masks the reference drew; tests/test_gpu_ref_fixtures.py)
mask_source = None
_mask_calls = 0


def drop_path_masks(drop_probs, B: int, device) -> Optional[torch.Tensor]:
    """All per-sample DropPath factors (mask / keep_prob, timm drop_path semantics: SURVEY A.2) of one forward pass in one
    launch: row r of the result belongs to ``drop_probs[r]``, rows in the order the reference draws them (block 0
    attention branch, block 0 MLP branch, block 1 ...).  Seeded from torch's CUDA generator seed (``torch.manual_seed``)
    plus a per-process call counter, so runs are reproducible without any device-side RNG state."""
    global _mask_calls
    if not any(p > 0.0 for p in drop_probs):
        return None
    if mask_source is not None:
        rs = mask_source(list(drop_probs), B, device)
        assert rs.shape == (len(drop_probs), B) and rs.dtype == torch.float32 and rs.is_cuda
        return rs.contiguous()
    rs = _empty((len(drop_probs), B), torch.float32, device)
    _mask_calls += 1
    L.droppath_masks(rs, drop_probs, torch.cuda.initial_seed(), _mask_calls)
    return rs


def drop_path_scale(drop_prob: float, training: bool, B: int, device) -> Optional[torch.Tensor]:
    """One DropPath's factor (stand-alone DropPath module)."""
    if drop_prob == 0.0 or not training:
        return None
    return drop_path_masks([drop_prob], B, device)[0]


# ================================================================================================
# Stand-alone leaf modules (the reference's own plug points: models/_compat.py:27-172).  The fused
# stages above bypass these inside a VisionTransformer; they exist so that Attention / Mlp /
# LayerNorm / PatchEmbed / nn.Linear-shaped heads are usable on their own, on the same kernels.
# All take and return fp32 (bf16 operands, fp32 accumulation inside).
# ================================================================================================
def _to_bf16(x: torch.Tensor) -> torch.Tensor:
    out = _empty(x.shape, torch.bfloat16, x.device)
    L.cast_bf16(x, out)
    return out


class LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, anchor, mod, store: ParamStore, save: bool):
        x = _require_f32_cuda(x, "LayerNorm input")
        D = x.shape[-1]
        rows = x.numel() // D
        y = _empty(x.shape, torch.bfloat16, x.device)
        mean, rstd = _empty((rows,), torch.float32, x.device), _empty((rows,), torch.float32, x.device)
        L.layernorm_fwd(x, mod.weight.data, mod.bias.data, y, mean, rstd, rows, D, mod.eps)
        if save:
            ctx.mod, ctx.store, ctx.saved = mod, store, (x, mean, rstd)
        return y.float()

    @staticmethod
    def backward(ctx, dy):
        mod, store = ctx.mod, ctx.store
        x, mean, rstd = ctx.saved
        ctx.saved = None
        D = x.shape[-1]
        rows = x.numel() // D
        dyb = _to_bf16(_require_f32_cuda(dy, "LayerNorm grad"))
        g = _empty(x.shape, torch.float32, x.device)
        L.layernorm_bwd(dyb, x, mean, rstd, mod.weight.data, None, g, None, None, 1, store.grad_of(mod.weight),
                        store.grad_of(mod.bias), rows, D)
        return g, None, None, None, None


class LinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, anchor, lin, store: ParamStore, save: bool):
        x = _require_f32_cuda(x, "Linear input")
        K, N = lin.in_features, lin.out_features
        M = x.numel() // K
        xb = _to_bf16(x)
        out = _empty(x.shape[:-1] + (N,), torch.float32, x.device)
        L.gemm(xb, store.shadow_of(lin.weight), out, M=M, N=N, K=K, epilogue=L.EPI_F32,
               bias=None if lin.bias is None else lin.bias.data)
        if save:
            ctx.lin, ctx.store, ctx.xb, ctx.shape = lin, store, xb, x.shape
        return out

    @staticmethod
    def backward(ctx, dy):
        lin, store, xb = ctx.lin, ctx.store, ctx.xb
        ctx.xb = None
        K, N = lin.in_features, lin.out_features
        M = xb.numel() // K
        dyb = _to_bf16(_require_f32_cuda(dy, "Linear grad"))
        L.gemm(dyb, xb, store.grad_of(lin.weight), M=N, N=K, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True,
               colsum=None if lin.bias is None else store.grad_of(lin.bias))
        dx = _empty(ctx.shape, torch.float32, dy.device)
        L.gemm(dyb, store.shadow_of(lin.weight), dx, M=M, N=K, K=N, epilogue=L.EPI_F32, b_mn=True)
        return dx, None, None, None, None


class AttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, anchor, attn, store: ParamStore, save: bool, attn_drop: float = 0.0):
        x = _require_f32_cuda(x, "Attention input")
        B, N, D = x.shape
        M, H, hd = B * N, attn.num_heads, attn.head_dim
        dev = x.device
        sh = store.shadow_of
        xb = _to_bf16(x).view(M, D)
        qkv = _empty((M, 3 * D), torch.bfloat16, dev)
        L.gemm(xb, sh(attn.qkv.weight), qkv, M=M, N=3 * D, K=D, epilogue=L.EPI_BF16,
               bias=None if attn.qkv.bias is None else attn.qkv.bias.data)
        att = _empty((M, D), torch.bfloat16, dev)
        lse = _empty((B, H, N), torch.float32, dev)
        ma = dropout_keep_mask("attn.attn_drop", B * H * N, N, attn_drop, dev)
        ascale = 1.0 / (1.0 - attn_drop) if ma is not None else 1.0
        L.attn_fwd(qkv, att, lse, B, N, H, hd, attn.scale, keep_mask=ma, keep_scale=ascale)
        out = _empty((B, N, D), torch.float32, dev)
        L.gemm(att, sh(attn.proj.weight), out, M=M, N=D, K=D, epilogue=L.EPI_F32,
               bias=None if attn.proj.bias is None else attn.proj.bias.data)
        if save:
            ctx.attn, ctx.store, ctx.saved, ctx.dims = attn, store, (xb, qkv, att, lse), (B, N, D, H, hd)
            ctx.adrop = (ma, ascale)
        return out

    @staticmethod
    def backward(ctx, dy):
        attn, store = ctx.attn, ctx.store
        xb, qkv, att, lse = ctx.saved
        ctx.saved = None
        B, N, D, H, hd = ctx.dims
        M = B * N
        dev = dy.device
        sh, gr = store.shadow_of, store.grad_of
        dyb = _to_bf16(_require_f32_cuda(dy, "Attention grad")).view(M, D)
        L.gemm(dyb, att, gr(attn.proj.weight), M=D, N=D, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True,
               colsum=None if attn.proj.bias is None else gr(attn.proj.bias))
        datt = _empty((M, D), torch.bfloat16, dev)
        L.gemm(dyb, sh(attn.proj.weight), datt, M=M, N=D, K=D, epilogue=L.EPI_BF16, b_mn=True)
        dqkv = _empty((M, 3 * D), torch.bfloat16, dev)
        L.attn_bwd(qkv, att, datt, lse, dqkv, B, N, H, hd, attn.scale, keep_mask=ctx.adrop[0], keep_scale=ctx.adrop[1])
        L.gemm(dqkv, xb, gr(attn.qkv.weight), M=3 * D, N=D, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True,
               colsum=None if attn.qkv.bias is None else gr(attn.qkv.bias))
        dx = _empty((B, N, D), torch.float32, dev)
        L.gemm(dqkv, sh(attn.qkv.weight), dx, M=M, N=D, K=3 * D, epilogue=L.EPI_F32, b_mn=True)
        return dx, None, None, None, None, None


class MlpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, anchor, mlp, store: ParamStore, save: bool, drop1: float = 0.0):
        x = _require_f32_cuda(x, "Mlp input")
        D, F, O = mlp.fc1.in_features, mlp.fc1.out_features, mlp.fc2.out_features
        M = x.numel() // D
        dev = x.device
        sh = store.shadow_of
        xb = _to_bf16(x).view(M, D)
        m1 = dropout_keep_mask("mlp.drop1", M, F, drop1, dev)
        h = _empty((M, F), torch.bfloat16, dev)
        act = _empty((M, F), torch.bfloat16, dev)
        L.gemm(xb, sh(mlp.fc1.weight), act, M=M, N=F, K=D, epilogue=L.EPI_GELU,
               bias=None if mlp.fc1.bias is None else mlp.fc1.bias.data, aux=h, mask=m1,
               mask_scale=1.0 / (1.0 - drop1) if m1 is not None else 1.0)
        out = _empty(x.shape[:-1] + (O,), torch.float32, dev)
        L.gemm(act, sh(mlp.fc2.weight), out, M=M, N=O, K=F, epilogue=L.EPI_F32,
               bias=None if mlp.fc2.bias is None else mlp.fc2.bias.data)
        if save:
            ctx.mlp, ctx.store, ctx.saved, ctx.shape = mlp, store, (xb, h, act), x.shape
        return out

    @staticmethod
    def backward(ctx, dy):
        mlp, store = ctx.mlp, ctx.store
        xb, h, act = ctx.saved
        ctx.saved = None
        D, F, O = mlp.fc1.in_features, mlp.fc1.out_features, mlp.fc2.out_features
        M = xb.numel() // D
        sh, gr = store.shadow_of, store.grad_of
        dyb = _to_bf16(_require_f32_cuda(dy, "Mlp grad")).view(M, O)
        L.gemm(dyb, act, gr(mlp.fc2.weight), M=O, N=F, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True,
               colsum=None if mlp.fc2.bias is None else gr(mlp.fc2.bias))
        dh = act
        L.gemm(dyb, sh(mlp.fc2.weight), dh, M=M, N=F, K=O, epilogue=L.EPI_DGELU, b_mn=True, aux=h)
        L.gemm(dh, xb, gr(mlp.fc1.weight), M=F, N=D, K=M, epilogue=L.EPI_ATOMIC, a_mn=True, b_mn=True,
               colsum=None if mlp.fc1.bias is None else gr(mlp.fc1.bias))
        dx = _empty(ctx.shape, torch.float32, dy.device)
        L.gemm(dh, sh(mlp.fc1.weight), dx, M=M, N=D, K=F, epilogue=L.EPI_F32, b_mn=True)
        return dx, None, None, None, None, None


class PatchEmbedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, anchor, pe, store: ParamStore, save: bool):
        img = _require_f32_cuda(img, "PatchEmbed input")
        B, C, H, W = img.shape
        ps = pe.patch_size[0]
        D = pe.proj.out_channels
        P, K = pe.num_patches, C * ps * ps
        patches = _empty((B * P, K), torch.bfloat16, img.device)
        L.patchify(img, patches, ps)
        out = _empty((B, P, D), torch.float32, img.device)
        L.gemm(patches, store.shadow_of(pe.proj.weight).view(D, K), out, M=B * P, N=D, K=K, epilogue=L.EPI_F32,
               bias=None if pe.proj.bias is None else pe.proj.bias.data)
        if save:
            ctx.pe, ctx.store, ctx.patches, ctx.dims = pe, store, patches, (B, P, D, K)
        return out

    @staticmethod
    def backward(ctx, dy):
        pe, store, patches = ctx.pe, ctx.store, ctx.patches
        ctx.patches = None
        B, P, D, K = ctx.dims
        dyb = _to_bf16(_require_f32_cuda(dy, "PatchEmbed grad")).view(B * P, D)
        L.gemm(dyb, patches, store.grad_of(pe.proj.weight).view(D, K), M=D, N=K, K=B * P, epilogue=L.EPI_ATOMIC,
               a_mn=True, b_mn=True, colsum=None if pe.proj.bias is None else store.grad_of(pe.proj.bias))
        return None, None, None, None, None
