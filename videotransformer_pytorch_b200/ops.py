"""Sub-block level autograd functions of the video-transformer hot path.

Each Function is the forward+backward of one reference sub-block, expressed as a fixed sequence of
C-ABI kernel launches (see _lib.K):

  TemporalAttnFn  <- DividedTemporalAttentionWithPreNorm.forward   (reference transformer.py:234-282)
  SpatialAttnFn   <- DividedSpatialAttentionWithPreNorm.forward    (transformer.py:336-382)
  JointAttnFn     <- MultiheadAttentionWithPreNorm.forward         (transformer.py:428-456)
  FFNFn           <- FFNWithPreNorm.forward                        (transformer.py:516-523)
  PatchTokensFn   <- PatchEmbed.forward + TimeSformer/ViViT.prepare_tokens
                     (transformer.py:138-151, video_transformer.py:193-240 / :455-475)
  PosEmbedInterpFn <- TimeSformer.interpolate_pos_encoding's bicubic F.interpolate (video_transformer.py:171-191)
  ClsNormFn       <- final nn.LayerNorm(eps=1e-6) + cls select     (video_transformer.py:251-254)
  AttentionCoreFn <- Attention.forward (stand-alone use)            (transformer.py:165-177)

Data layout: the residual stream stays fp32 `[B, 1+P*T, D]` exactly as in the reference (token
n = 1 + p*T + t).  The einops regroupings ('b (p t) d -> (b p) t d', '-> (b t) p d', cls replication /
mean) never materialise: LayerNorm reads rows through an index map and the last GEMM of each
sub-block scatters rows back through the inverse map while adding the residual.  GEMM operands are
bf16 (fp32 accumulation in TMEM); weights are bf16 shadows of the fp32 nn.Parameters.
"""
from __future__ import annotations

import functools

import torch

from . import _lib


def K():
    return _lib.K


_MASK_ARENA = None

# FFN activation: fused into the FC1 / FC2-dgrad GEMM epilogues (VT_EPI_GELU / VT_EPI_DGELU) or as stand-alone
# bandwidth kernels after a plain bf16 epilogue.  Round 1 measured the split form faster (the erf math sat in the slow
# transposing epilogue); the forward GELU epilogue now stores z and h as two TMA boxes — VT_FUSED_GELU=1 selects it
# for FC1 (the dGELU epilogue of the FC2 data gradient stays split).
import os as _os
FUSED_GELU_FWD = _os.environ.get('VT_FUSED_GELU', '0') == '1'
FUSED_DGELU_BWD = _os.environ.get('VT_TMA_DGELU', '0') == '1'      # dGELU epilogue of the FC2 data gradient on TMA
FUSED_GELU_EPILOGUE = False
# bias gradients from the kernels that produce dY (gather_cast / dgelu with column sums) instead of a separate pass;
# VT_FUSED_COLSUM=0/1 overrides
FUSED_COLSUM = _os.environ.get('VT_FUSED_COLSUM', '1') == '1'
# temporal_fc(DropPath(proj(.))) as ONE token GEMM with the product weight W_fc W_proj (two 768^3 GEMMs per step instead of
# two 12544 x 768 x 768 ones forward, and the same saving twice in backward); VT_MERGE_TEMPORAL_FC=0/1 overrides
MERGE_TEMPORAL_FC = _os.environ.get('VT_MERGE_TEMPORAL_FC', '1') == '1'


def set_mask_arena(arena):
    """Installed by graph.GraphedTrainStep while a step is being captured."""
    global _MASK_ARENA
    _MASK_ARENA = arena


# --------------------------------------------------------------------------------------------------
# index maps (int32, cached per geometry/device)
# --------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=64)
def token_maps(B: int, T: int, P: int, device: str):
    dev = torch.device(device)
    S = 1 + P * T
    R = B * S
    ar = functools.partial(torch.arange, device=dev, dtype=torch.int64)
    # temporal layout m = (b*P + p)*T + t  ==  patch rows of the residual stream in order
    m = ar(B * P * T)
    temporal = (m // (P * T)) * S + 1 + (m % (P * T))
    # spatial layout m = (b*T + t)*(P+1) + n ; n = 0 -> cls of sample b, n >= 1 -> patch n-1 of frame t
    m = ar(B * T * (P + 1))
    bt, n = m // (P + 1), m % (P + 1)
    b, t = bt // T, bt % T
    is_cls = n == 0
    src = torch.where(is_cls, b * S, b * S + 1 + (n - 1) * T + t)
    sp_out = torch.where(is_cls, R + bt, src)                 # forward: cls outputs go to R + (b*T+t)
    sp_aux = torch.where(is_cls, torch.full_like(src, -1), src)
    sp_bwd = torch.where(is_cls, -(bt) - 1, src)              # LN backward: cls grads go to aux[b*T+t]
    cls_scale = torch.where(is_cls, torch.full_like(src, 1.0, dtype=torch.float32) / T,
                            torch.ones_like(src, dtype=torch.float32))
    # patch-embed GEMM rows m = (b*T + t)*P + p
    m = ar(B * T * P)
    bt, p = m // P, m % P
    b, t = bt // T, bt % T
    emb_out = b * S + 1 + p * T + t
    emb_aux = p * T + t
    i32 = lambda v: v.to(torch.int32).contiguous()
    return dict(temporal=i32(temporal), sp_in=i32(src), sp_out=i32(sp_out), sp_aux=i32(sp_aux), sp_bwd=i32(sp_bwd),
                sp_cls_scale=cls_scale.contiguous(), emb_out=i32(emb_out), emb_aux=i32(emb_aux),
                cls_rows=i32(ar(B) * S))


def affine_row_maps(B: int, T: int, P: int, D: int):
    """The temporal / spatial row maps of token_maps() in closed form (vt_gemm_params.map_*): GEMM row m has outer = m // period,
    inner = m % period and lands at element  base + (outer % tcount) * stride_t + (inner - skip) * stride_p +
    (outer // tcount) * stride_b  of the [B*(1+P*T) (+B*T), D] residual stream; `skip` leading rows of every period are the
    replicated cls rows of the spatial pass, written to the B*T side rows after the stream."""
    S = 1 + P * T
    temporal = dict(period=P * T, skip=0, tcount=1, stride_t=D, stride_p=D, stride_b=S * D, base=D)
    spatial = dict(period=P + 1, skip=1, tcount=T, stride_t=D, stride_p=T * D, stride_b=S * D, base=D,
                   special_base=B * S * D, special_stride=D)
    return dict(temporal=temporal, spatial=spatial)


@functools.lru_cache(maxsize=64)
def frame_maps(BT: int, P: int, device: str):
    """ViViT spatial encoder tokens: rows (bt, n); patch-embed GEMM rows (bt, p) -> bt*(P+1)+1+p."""
    dev = torch.device(device)
    m = torch.arange(BT * P, device=dev, dtype=torch.int64)
    bt, p = m // P, m % P
    out = bt * (P + 1) + 1 + p
    aux = 1 + p
    return dict(emb_out=out.to(torch.int32).contiguous(), emb_aux=aux.to(torch.int32).contiguous())


def drop_path_scale(p: float, training: bool, n0: int, repeat: int, device):
    """Per-row DropPath factor, reference transformer.py:34-42: mask = floor(keep + U[0,1)) drawn with
    torch.rand on the CPU default generator (one value per dim-0 row of the sub-block's own layout),
    output = x / keep * mask.  Returns fp32 [n0*repeat] on `device`, or None when DropPath is inactive."""
    if p == 0.0 or not training:
        return None
    keep = 1.0 - p
    if _MASK_ARENA is not None and _MASK_ARENA.recording:
        # CUDA-graph capture (graph.py): the factors live in a static arena refilled before every replay;
        # only the expansion to per-row granularity is part of the graph.
        r = _MASK_ARENA.register(n0, keep)
        return r.repeat_interleave(repeat).contiguous() if repeat > 1 else r.contiguous()
    r = (keep + torch.rand((n0, 1, 1))).floor_().reshape(n0) / keep
    r = r.to(device=device, dtype=torch.float32, non_blocking=True)
    return r.repeat_interleave(repeat).contiguous() if repeat > 1 else r.contiguous()


# While a data-parallel step is being captured (graph.GraphedTrainStep with ddp.GradientBuckets) this maps the address of a
# weight parameter to its slice of the flat gradient bucket: the weight-gradient GEMM then writes (zero + split-K TMA
# reduce-add) straight into the bucket and no gather copy precedes the all-reduce (SURVEY C1).  Never set in eager mode,
# where autograd ACCUMULATES the returned gradient into p.grad — returning p.grad's own storage would double it.
GRAD_DEST = None
GRAD_DEST_ZEROED = False


def set_grad_destinations(table, zeroed=False):
    """table: {parameter data_ptr: fp32 view the weight-gradient GEMM of that parameter writes to} or None.
    zeroed: the views were zeroed after the previous backward (one memset of the arena / buckets per step), so the split-K
    GEMMs skip their own per-output memset."""
    global GRAD_DEST, GRAD_DEST_ZEROED
    GRAD_DEST = table
    GRAD_DEST_ZEROED = bool(zeroed) and table is not None


def _wgrad(dout, act, n_out, k_in, m_tok, tag=None, wptr=None):
    """dW[n_out, k_in] = dout[m_tok, n_out]^T @ act[m_tok, k_in]  (both operands MN-major, split-K).
    wptr: data_ptr() of the fp32 parameter this is the gradient of (see GRAD_DEST)."""
    out = _grad_dest(wptr, n_out, k_in)
    return K().gemm(dout, act, n_out, k_in, m_tok, a_mn=True, b_mn=True, epi='f32', split_ok=True, tag=tag, out=out,
                    out_zeroed=out is not None and GRAD_DEST_ZEROED)


def _grad_dest(wptr, n_out, k_in):
    """The DDP bucket slice registered for the parameter at wptr (GRAD_DEST), as an [n_out, k_in] view, or None."""
    if GRAD_DEST is None or wptr is None:
        return None
    dest = GRAD_DEST.get(wptr)
    if dest is not None and dest.numel() == n_out * k_in and dest.is_contiguous() and dest.data_ptr() % 16 == 0 and k_in % 4 == 0:
        return dest.view(n_out, k_in)          # TMA stores need a 16-byte aligned base and row pitch
    return None


def _dgrad(dout, w, m_tok, k_in, n_out, **kw):
    """dX[m_tok, k_in] = dout[m_tok, n_out] @ W[n_out, k_in]  (W read MN-major)."""
    return K().gemm(dout, w, m_tok, k_in, n_out, b_mn=True, **kw)


ATTN_SINGLE_PASS_MAX = 256      # vt_attn_*: whole score row in TMEM / registers; longer sequences stream K/V (vt_xattn_*)


def _packed_heads(qkv, Bp, N, H, hd):
    """q, k, v of a packed [Bp*N, 3*H*hd] projection as [Bp, H, N, hd] views (token-major, no copy)."""
    v5 = qkv.view(Bp, N, 3, H, hd)
    return tuple(v5[:, :, s].permute(0, 2, 1, 3) for s in range(3))


def _streaming_attn_bwd(k, qkv, cx, dcx, lse, Bp, N, H, hd):
    """dqkv of a long-sequence attention through the streaming tcgen05 kernels (q/k/v and dq in place in the packed layout)."""
    q4, k4, v4 = _packed_heads(qkv, Bp, N, H, hd)
    dqkv = torch.empty_like(qkv)
    dq4, dk4, dv4 = _packed_heads(dqkv, Bp, N, H, hd)
    D = H * hd
    dk, dv = k.xattn_bwd(q4, k4, v4, cx.view(Bp, N, D), dcx.view(Bp, N, D), lse, hd ** -0.5, dq4)
    dk4.copy_(dk)           # fp32 [Bp,H,N,hd] accumulators -> their bf16 slots of the packed gradient
    dv4.copy_(dv)
    return dqkv


def _cast_with_colsum(k, src2d, in_row=None, row_scale=None, rows=None):
    """dY in bf16 (gathered / scaled rows of the fp32 gradient stream) and its column sums = the bias gradient."""
    if FUSED_COLSUM:
        return k.gather_cast_colsum(src2d, in_row=in_row, row_scale=row_scale, rows=rows)
    g = k.gather_cast(src2d, in_row=in_row, row_scale=row_scale, rows=rows)
    return g, k.colsum(g)


def _mul_opt(a, b):
    if a is None:
        return b
    if b is None:
        return a
    return a * b


# --------------------------------------------------------------------------------------------------
class TemporalAttnFn(torch.autograd.Function):
    """y = cat(cls, x_p + temporal_fc(DropPath(proj(attn_T(LN(x_p))))))."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, qkv_w, qkv_b, proj_w, proj_b, fc_w, fc_b, qkv_wh, proj_wh, fc_wh, dp, T, H, eps=1e-5):
        k = K()
        B, S, D = x.shape
        P = (S - 1) // T
        maps = token_maps(B, T, P, str(x.device))
        x2 = x.reshape(B * S, D)
        Mt = B * P * T
        xn, mean, rstd = k.ln_fwd(x2, ln_w, ln_b, eps, in_row=maps['temporal'], rows=Mt)
        qkv = k.gemm(xn, qkv_wh, Mt, 3 * D, D, bias=qkv_b, epi='bf16', tag='qkv')
        hd = D // H
        cx, lse, _ = k.attn_fwd(qkv, B * P, T, H, hd, hd ** -0.5)
        y = torch.empty_like(x)
        y2 = y.view(B * S, D)
        ctx.merged = MERGE_TEMPORAL_FC
        if ctx.merged:
            # y = s (W_f (W_p c + b_p)) + b_f + x = s (W_c c + b_c) + b_f + x,  W_c = W_f W_p,  b_c = W_f b_p
            # (transformer.py:261-267: two nn.Linear with only DropPath's per-sample scale between them)
            wc = k.gemm(fc_wh, proj_wh, D, D, D, b_mn=True, epi='bf16')
            bc = torch.mv(fc_w.detach().float(), proj_b.detach().float())
            k.gemm(cx, wc, Mt, D, D, bias=bc, bias2=fc_b, epi='f32', aux=x2, aux_row=maps['temporal'], out=y2,
                   out_row=maps['temporal'], row_scale=dp, row_map=affine_row_maps(B, T, P, D)['temporal'], tag='proj')
            a = wc
        else:
            a = k.gemm(cx, proj_wh, Mt, D, D, bias=proj_b, epi='bf16', row_scale=dp, tag='proj')
            k.gemm(a, fc_wh, Mt, D, D, bias=fc_b, epi='f32', aux=x2, aux_row=maps['temporal'], out=y2,
                   out_row=maps['temporal'], row_map=affine_row_maps(B, T, P, D)['temporal'])
        k.cls_rows(y[:, 0], x[:, 0])
        ctx.save_for_backward(x, ln_w, mean, rstd, xn, qkv, cx, lse, a, qkv_wh, proj_wh, fc_wh, dp,
                              fc_w if ctx.merged else None, proj_b if ctx.merged else None)
        ctx.geom = (B, S, D, T, H, P)
        ctx.wptrs = (qkv_w.data_ptr(), proj_w.data_ptr(), fc_w.data_ptr())
        return y

    @staticmethod
    def backward(ctx, dy):
        k = K()
        x, ln_w, mean, rstd, xn, qkv, cx, lse, a, qkv_wh, proj_wh, fc_wh, dp, fc_w, proj_b = ctx.saved_tensors
        B, S, D, T, H, P = ctx.geom
        maps = token_maps(B, T, P, str(x.device))
        hd = D // H
        Mt = B * P * T
        dy = dy.contiguous()
        dy2 = dy.view(B * S, D)
        x2 = x.reshape(B * S, D)
        if ctx.merged:
            # gs = s * dY rows;  v = colsum(gs);  G = gs^T c
            # dc = gs W_c;  dW_f = G W_p^T + v b_p^T;  db_f = colsum(dY);  dW_p = W_f^T G;  db_p = W_f^T v
            wc = a
            if dp is None:
                gs, v = _cast_with_colsum(k, dy2, in_row=maps['temporal'], rows=Mt)
                d_fc_b = v
            elif FUSED_COLSUM:
                gs, v, d_fc_b = k.gather_cast_colsum(dy2, in_row=maps['temporal'], row_scale=dp, rows=Mt, unscaled_sums=True)
            else:
                gs = k.gather_cast(dy2, in_row=maps['temporal'], row_scale=dp, rows=Mt)
                v = k.colsum(gs)
                d_fc_b = k.colsum(k.gather_cast(dy2, in_row=maps['temporal'], rows=Mt))
            dcx = _dgrad(gs, wc, Mt, D, D, epi='bf16', tag='proj')
            G = k.gemm(gs, cx, D, D, Mt, a_mn=True, b_mn=True, epi='f32', split_ok=True, tag='proj')
            Gh = k.cast_bf16(G)
            d_fc_w = k.gemm(Gh, proj_wh, D, D, D, epi='f32', out=_grad_dest(ctx.wptrs[2], D, D))
            d_fc_w.addr_(v, proj_b.detach().float())
            d_proj_w = k.gemm(fc_wh, Gh, D, D, D, a_mn=True, b_mn=True, epi='f32', out=_grad_dest(ctx.wptrs[1], D, D))
            d_proj_b = torch.mv(fc_w.detach().float().t(), v)
        else:
            g, d_fc_b = _cast_with_colsum(k, dy2, in_row=maps['temporal'], rows=Mt)
            d_fc_w = _wgrad(g, a, D, D, Mt, wptr=ctx.wptrs[2])
            da = _dgrad(g, fc_wh, Mt, D, D, epi='bf16', row_scale=dp)
            d_proj_w = _wgrad(da, cx, D, D, Mt, tag='proj', wptr=ctx.wptrs[1])
            d_proj_b = k.colsum(da)
            dcx = _dgrad(da, proj_wh, Mt, D, D, epi='bf16', tag='proj')
        dqkv = k.attn_bwd(qkv, cx, dcx, lse, B * P, T, H, hd, hd ** -0.5)
        d_qkv_w = _wgrad(dqkv, xn, 3 * D, D, Mt, tag='qkv', wptr=ctx.wptrs[0])
        d_qkv_b = k.colsum(dqkv)
        dxn = _dgrad(dqkv, qkv_wh, Mt, D, 3 * D, epi='bf16', tag='qkv')
        dx = torch.empty_like(x)
        _, _, d_ln_w, d_ln_b = k.ln_bwd(dxn, x2, mean, rstd, ln_w, in_row=maps['temporal'], out_row=maps['temporal'],
                                        dres=dy2, dx=dx.view(B * S, D))
        k.cls_rows(dx[:, 0], dy[:, 0])
        return (dx, d_ln_w, d_ln_b, d_qkv_w, d_qkv_b, d_proj_w, d_proj_b, d_fc_w, d_fc_b,
                None, None, None, None, None, None, None)


# --------------------------------------------------------------------------------------------------
class SpatialAttnFn(torch.autograd.Function):
    """y = x + cat(mean_t(cls_out), patches_out), out = DropPath(proj(attn_{1+P}(LN(cat(cls, frame)))))."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, qkv_w, qkv_b, proj_w, proj_b, qkv_wh, proj_wh, dp, T, H, eps=1e-5):
        k = K()
        B, S, D = x.shape
        P = (S - 1) // T
        maps = token_maps(B, T, P, str(x.device))
        R, Ms = B * S, B * T * (P + 1)
        x2 = x.reshape(R, D)
        hd = D // H
        xn, mean, rstd = k.ln_fwd(x2, ln_w, ln_b, eps, in_row=maps['sp_in'], rows=Ms)
        qkv = k.gemm(xn, qkv_wh, Ms, 3 * D, D, bias=qkv_b, epi='bf16', tag='qkv')
        if P + 1 <= ATTN_SINGLE_PASS_MAX:
            cx, lse, _ = k.attn_fwd(qkv, B * T, P + 1, H, hd, hd ** -0.5)
        else:
            # frames past 16 x 16 patches (img_size >= 256 at patch 16): streaming tcgen05 kernel, q/k/v read in place
            q4, k4, v4 = _packed_heads(qkv, B * T, P + 1, H, hd)
            cx, lse = k.xattn_fwd(q4, k4, v4, hd ** -0.5)
            cx = cx.view(Ms, D)
        ybig = torch.empty((R + B * T, D), dtype=torch.float32, device=x.device)
        k.gemm(cx, proj_wh, Ms, D, D, bias=proj_b, epi='f32', aux=x2, aux_row=maps['sp_aux'], out=ybig,
               out_row=maps['sp_out'], row_scale=dp, row_map=affine_row_maps(B, T, P, D)['spatial'], tag='proj')
        y = ybig[:R].view(B, S, D)
        k.cls_rows(y[:, 0], x[:, 0], extra=ybig[R:].view(B, T, D), scale=1.0 / T)
        ctx.save_for_backward(x, ln_w, mean, rstd, xn, qkv, cx, lse, qkv_wh, proj_wh, dp)
        ctx.geom = (B, S, D, T, H, P)
        ctx.wptrs = (qkv_w.data_ptr(), proj_w.data_ptr())
        return y

    @staticmethod
    def backward(ctx, dy):
        k = K()
        x, ln_w, mean, rstd, xn, qkv, cx, lse, qkv_wh, proj_wh, dp = ctx.saved_tensors
        B, S, D, T, H, P = ctx.geom
        maps = token_maps(B, T, P, str(x.device))
        hd = D // H
        R, Ms = B * S, B * T * (P + 1)
        dy = dy.contiguous()
        dy2 = dy.view(R, D)
        x2 = x.reshape(R, D)
        g, d_proj_b = _cast_with_colsum(k, dy2, in_row=maps['sp_in'], row_scale=_mul_opt(dp, maps['sp_cls_scale']), rows=Ms)
        d_proj_w = _wgrad(g, cx, D, D, Ms, tag='proj', wptr=ctx.wptrs[1])
        dcx = _dgrad(g, proj_wh, Ms, D, D, epi='bf16', tag='proj')
        if P + 1 <= ATTN_SINGLE_PASS_MAX:
            dqkv = k.attn_bwd(qkv, cx, dcx, lse, B * T, P + 1, H, hd, hd ** -0.5)
        else:
            dqkv = _streaming_attn_bwd(k, qkv, cx, dcx, lse, B * T, P + 1, H, hd)
        d_qkv_w = _wgrad(dqkv, xn, 3 * D, D, Ms, tag='qkv', wptr=ctx.wptrs[0])
        d_qkv_b = k.colsum(dqkv)
        dxn = _dgrad(dqkv, qkv_wh, Ms, D, 3 * D, epi='bf16', tag='qkv')
        dx = torch.empty_like(x)
        _, aux, d_ln_w, d_ln_b = k.ln_bwd(dxn, x2, mean, rstd, ln_w, in_row=maps['sp_in'], out_row=maps['sp_bwd'],
                                          dres=dy2, dx=dx.view(R, D), n_aux=B * T)
        k.cls_rows(dx[:, 0], dy[:, 0], extra=aux.view(B, T, D))
        return dx, d_ln_w, d_ln_b, d_qkv_w, d_qkv_b, d_proj_w, d_proj_b, None, None, None, None, None, None


# --------------------------------------------------------------------------------------------------
class JointAttnFn(torch.autograd.Function):
    """y = x + DropPath(proj(attn_N(LN(x)))) on [Bp, N, D]."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, qkv_w, qkv_b, proj_w, proj_b, qkv_wh, proj_wh, dp, H, eps=1e-5):
        k = K()
        Bp, N, D = x.shape
        M = Bp * N
        x2 = x.reshape(M, D)
        hd = D // H
        xn, mean, rstd = k.ln_fwd(x2, ln_w, ln_b, eps)
        qkv = k.gemm(xn, qkv_wh, M, 3 * D, D, bias=qkv_b, epi='bf16', tag='qkv')
        if N <= ATTN_SINGLE_PASS_MAX:
            cx, lse, _ = k.attn_fwd(qkv, Bp, N, H, hd, hd ** -0.5)
        else:
            # long sequences (joint space-time attention: 1 + P*T = 1569 tokens): streaming tcgen05 kernel, q/k/v read in
            # place from the packed projection
            q4, k4, v4 = _packed_heads(qkv, Bp, N, H, hd)
            cx, lse = k.xattn_fwd(q4, k4, v4, hd ** -0.5)
            cx = cx.view(M, D)
        y = torch.empty_like(x)
        k.gemm(cx, proj_wh, M, D, D, bias=proj_b, epi='f32', aux=x2, out=y.view(M, D), row_scale=dp, tag='proj')
        ctx.save_for_backward(x, ln_w, mean, rstd, xn, qkv, cx, lse, qkv_wh, proj_wh, dp)
        ctx.geom = (Bp, N, D, H)
        ctx.wptrs = (qkv_w.data_ptr(), proj_w.data_ptr())
        return y

    @staticmethod
    def backward(ctx, dy):
        k = K()
        x, ln_w, mean, rstd, xn, qkv, cx, lse, qkv_wh, proj_wh, dp = ctx.saved_tensors
        Bp, N, D, H = ctx.geom
        hd = D // H
        M = Bp * N
        dy = dy.contiguous()
        dy2 = dy.view(M, D)
        x2 = x.reshape(M, D)
        g, d_proj_b = _cast_with_colsum(k, dy2, row_scale=dp)
        d_proj_w = _wgrad(g, cx, D, D, M, tag='proj', wptr=ctx.wptrs[1])
        dcx = _dgrad(g, proj_wh, M, D, D, epi='bf16', tag='proj')
        if N <= ATTN_SINGLE_PASS_MAX:
            dqkv = k.attn_bwd(qkv, cx, dcx, lse, Bp, N, H, hd, hd ** -0.5)
        else:
            dqkv = _streaming_attn_bwd(k, qkv, cx, dcx, lse, Bp, N, H, hd)
        d_qkv_w = _wgrad(dqkv, xn, 3 * D, D, M, tag='qkv', wptr=ctx.wptrs[0])
        d_qkv_b = k.colsum(dqkv)
        dxn = _dgrad(dqkv, qkv_wh, M, D, 3 * D, epi='bf16', tag='qkv')
        dx = torch.empty_like(x)
        _, _, d_ln_w, d_ln_b = k.ln_bwd(dxn, x2, mean, rstd, ln_w, dres=dy2, dx=dx.view(M, D))
        return dx, d_ln_w, d_ln_b, d_qkv_w, d_qkv_b, d_proj_w, d_proj_b, None, None, None, None, None


# --------------------------------------------------------------------------------------------------
class FFNFn(torch.autograd.Function):
    """y = x + DropPath(W2 gelu(W1 LN(x) + b1) + b2) on [B, S, D]."""

    @staticmethod
    def forward(ctx, x, ln_w, ln_b, w1, b1, w2, b2, w1h, w2h, dp, eps=1e-5):
        k = K()
        D = x.shape[-1]
        M = x.numel() // D
        Dh = w1h.shape[0]
        x2 = x.reshape(M, D)
        xn, mean, rstd = k.ln_fwd(x2, ln_w, ln_b, eps)
        if FUSED_GELU_EPILOGUE or FUSED_GELU_FWD:
            z, h = k.gemm(xn, w1h, M, Dh, D, bias=b1, epi='gelu')
        else:
            z = k.gemm(xn, w1h, M, Dh, D, bias=b1, epi='bf16')
            h = k.gelu(z)
        y = torch.empty_like(x)
        k.gemm(h, w2h, M, D, Dh, bias=b2, epi='f32', aux=x2, out=y.view(M, D), row_scale=dp)
        ctx.save_for_backward(x, ln_w, mean, rstd, xn, z, h, w1h, w2h, dp)
        ctx.wptrs = (w1.data_ptr(), w2.data_ptr())
        return y

    @staticmethod
    def backward(ctx, dy):
        k = K()
        x, ln_w, mean, rstd, xn, z, h, w1h, w2h, dp = ctx.saved_tensors
        D = x.shape[-1]
        M = x.numel() // D
        Dh = w1h.shape[0]
        dy = dy.contiguous()
        dy2 = dy.view(M, D)
        x2 = x.reshape(M, D)
        g, d_b2 = _cast_with_colsum(k, dy2, row_scale=dp)
        d_w2 = _wgrad(g, h, D, Dh, M, wptr=ctx.wptrs[1])
        d_b1 = None
        if FUSED_GELU_EPILOGUE or FUSED_DGELU_BWD:
            dz = _dgrad(g, w2h, M, Dh, D, epi='dgelu', aux=z)
        else:
            if FUSED_COLSUM:
                dz, d_b1 = k.dgelu_colsum(_dgrad(g, w2h, M, Dh, D, epi='bf16'), z)
            else:
                dz = k.dgelu(_dgrad(g, w2h, M, Dh, D, epi='bf16'), z)
        d_w1 = _wgrad(dz, xn, Dh, D, M, wptr=ctx.wptrs[0])
        if d_b1 is None:
            d_b1 = k.colsum(dz)
        dxn = _dgrad(dz, w1h, M, D, Dh, epi='bf16')
        dx = torch.empty_like(x)
        _, _, d_ln_w, d_ln_b = k.ln_bwd(dxn, x2, mean, rstd, ln_w, dres=dy2, dx=dx.view(M, D))
        return dx, d_ln_w, d_ln_b, d_w1, d_b1, d_w2, d_b2, None, None, None, None


# --------------------------------------------------------------------------------------------------
class PatchTokensFn(torch.autograd.Function):
    """Patch / tubelet projection fused with token assembly.

    mode 'timesformer': out [B, 1+P*T, D], row 1+p*T+t = conv(x)[b,t,p] + pos[1+p] + time[t];
                        row 0 = cls + pos[0]                     (video_transformer.py:199-237)
    mode 'frames'     : out [B*T', 1+P, D], row 1+p = conv(x)[bt,p] + pos[1+p]; row 0 = cls + pos[0]
                        (ViViT fact_encoder, video_transformer.py:461-471)
    """

    @staticmethod
    def forward(ctx, x, w, b, cls_token, pos_embed, time_embed, wh, mode, tube, norm=None, mix_plan=None):
        k = K()
        D = w.shape[0]
        ph, pw = w.shape[-2], w.shape[-1]
        if x.dtype == torch.uint8:
            # decoder output [B, T, H, W, C]: ToTensor + Normalize are folded into the operand kernel (norm = (scale, shift)),
            # and with a mix plan (mixup.Mixup) the batch-level Mixup / CutMix of mixup.py:102-114 as well
            B, T, Himg, Wimg, C = x.shape
            if mix_plan is not None:
                cols = k.im2col_u8_mix(x, norm[0], norm[1], mix_plan, tube, ph, pw)
            else:
                cols = k.im2col_u8(x, norm[0], norm[1], tube, ph, pw)
        else:
            B, T, C, Himg, Wimg = x.shape
            cols = k.im2col(x.float(), tube, ph, pw)
        Tp = T // tube
        P = (Himg // ph) * (Wimg // pw)
        Kc = C * tube * ph * pw
        M = B * Tp * P
        pos = pos_embed.reshape(-1, D).float()
        if mode == 'timesformer':
            maps = token_maps(B, Tp, P, str(x.device))
            S = 1 + P * Tp
            table = (pos[1:, None, :] + time_embed.reshape(-1, D).float()[None, :, :]).reshape(P * Tp, D).contiguous()
            out = torch.empty((B, S, D), dtype=torch.float32, device=x.device)
            out_row, aux_row = maps['emb_out'], maps['emb_aux']
        else:
            maps = frame_maps(B * Tp, P, str(x.device))
            S = 1 + P
            table = pos.contiguous()
            out = torch.empty((B * Tp, S, D), dtype=torch.float32, device=x.device)
            out_row, aux_row = maps['emb_out'], maps['emb_aux']
        k.gemm(cols, wh.reshape(D, Kc), M, D, Kc, bias=b, epi='f32', aux=table, aux_row=aux_row,
               out=out.view(-1, D), out_row=out_row)
        out[:, 0] = cls_token.reshape(D).float() + pos[0]
        ctx.save_for_backward(cols, wh)
        ctx.meta = (mode, tube, (B, T, C, Himg, Wimg), tuple(w.shape), tuple(cls_token.shape), tuple(pos_embed.shape),
                    None if time_embed is None else tuple(time_embed.shape), P, Tp,
                    ctx.needs_input_grad[0] and x.dtype != torch.uint8)
        return out

    @staticmethod
    def backward(ctx, dout):
        k = K()
        cols, wh = ctx.saved_tensors
        mode, tube, xshape, wshape, cshape, pshape, tshape, P, Tp, need_dx = ctx.meta
        B = xshape[0]
        D = wshape[0]
        Kc = cols.shape[1]
        M = cols.shape[0]
        dout = dout.contiguous()
        d2 = dout.view(-1, D)
        if mode == 'timesformer':
            maps = token_maps(B, Tp, P, str(dout.device))
        else:
            maps = frame_maps(B * Tp, P, str(dout.device))
        g, db = _cast_with_colsum(k, d2, in_row=maps['emb_out'], rows=M)
        dw = _wgrad(g, cols, D, Kc, M).view(wshape)
        dcls = dout[:, 0].sum(dim=0)
        if mode == 'timesformer':
            dtab = dout[:, 1:].sum(dim=0).view(P, Tp, D)
            dpos = torch.cat((dcls[None], dtab.sum(dim=1)), dim=0).view(pshape)
            dtime = dtab.sum(dim=0).reshape(tshape).clone()
        else:
            dpos = torch.cat((dcls[None], dout[:, 1:].sum(dim=0)), dim=0).view(pshape)
            dtime = None
        dx = None
        if need_dx:
            dcols = _dgrad(g, wh.reshape(D, Kc), M, Kc, D, epi='f32')
            dx = k.col2im(dcols, xshape, tube, wshape[-2], wshape[-1])
        # small grads are returned as fresh contiguous tensors (not views) so autograd can adopt them in place
        return dx, dw.contiguous(), db, dcls.reshape(cshape).clone(), dpos.contiguous(), dtime, None, None, None, None, None


# --------------------------------------------------------------------------------------------------
class PosEmbedInterpFn(torch.autograd.Function):
    """Bicubic resampling of the spatial position table [1, 1+side^2, D] -> [1, 1+rows*cols, D] (cls row copied), the
    F.interpolate of TimeSformer.interpolate_pos_encoding (video_transformer.py:184-191); scale_r / scale_c are the inverse
    scale factors.  Backward is the kernel's adjoint."""

    @staticmethod
    def forward(ctx, pos, side, rows, cols, scale_r, scale_c):
        D = pos.shape[-1]
        out = K().pos_interp_fwd(pos.reshape(-1, D).float().contiguous(), side, rows, cols, scale_r, scale_c)
        ctx.geom = (tuple(pos.shape), side, rows, cols, scale_r, scale_c)
        return out.view(1, 1 + rows * cols, D)

    @staticmethod
    def backward(ctx, dout):
        pshape, side, rows, cols, scale_r, scale_c = ctx.geom
        d = K().pos_interp_bwd(dout.reshape(-1, pshape[-1]).float().contiguous(), side, rows, cols, scale_r, scale_c)
        return d.view(pshape), None, None, None, None, None


# --------------------------------------------------------------------------------------------------
class RowsNormFn(torch.autograd.Function):
    """fp32 LayerNorm of selected rows of x2d [R, D] -> [len(rows), D] (final norm on the rows that are
    actually consumed, video_transformer.py:251-256; rows=None => all rows)."""

    @staticmethod
    def forward(ctx, x, w, b, eps, rows):
        k = K()
        D = x.shape[-1]
        x2 = x.reshape(-1, D)
        n = x2.shape[0] if rows is None else rows.numel()
        y, mean, rstd = k.ln_fwd(x2, w, b, eps, in_row=rows, rows=n, out_fp32=True)
        ctx.save_for_backward(x, w, mean, rstd, rows if rows is not None else torch.empty(0))
        ctx.has_rows = rows is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        k = K()
        x, w, mean, rstd, rows = ctx.saved_tensors
        rows = rows if ctx.has_rows else None
        D = x.shape[-1]
        x2 = x.reshape(-1, D)
        dx = torch.zeros_like(x) if rows is not None else torch.empty_like(x)
        _, _, dw, db = k.ln_bwd(dy.contiguous().float(), x2, mean, rstd, w, in_row=rows, out_row=rows,
                                dx=dx.view(-1, D))
        return dx, dw, db, None, None


# --------------------------------------------------------------------------------------------------
class AttentionCoreFn(torch.autograd.Function):
    """Stand-alone Attention.forward (transformer.py:165-177): qkv linear, softmax(qk^T*scale)v, proj.
    Returns (out fp32 [Bp,N,C], probs fp32 [Bp,H,N,N]); probs is not differentiable."""

    @staticmethod
    def forward(ctx, x, qkv_w, qkv_b, proj_w, proj_b, qkv_wh, proj_wh, H, want_probs):
        k = K()
        Bp, N, C = x.shape
        M = Bp * N
        hd = C // H
        xh = k.gather_cast(x.reshape(M, C).float().contiguous())
        qkv = k.gemm(xh, qkv_wh, M, 3 * C, C, bias=qkv_b, epi='bf16')
        if N <= ATTN_SINGLE_PASS_MAX:
            cx, lse, probs = k.attn_fwd(qkv, Bp, N, H, hd, hd ** -0.5, want_probs=want_probs)
        else:
            # long sequences (joint space-time: 1569 tokens): context by the streaming tcgen05 kernel; the probability
            # maps the reference returns (transformer.py:171-177) by a row-tile softmax kernel, 8 query rows per CTA
            q4, k4, v4 = _packed_heads(qkv, Bp, N, H, hd)
            cx, lse = k.xattn_fwd(q4, k4, v4, hd ** -0.5)
            cx = cx.view(M, C)
            probs = k.attn_probs(qkv, Bp, N, H, hd, hd ** -0.5) if want_probs else None
        out = k.gemm(cx, proj_wh, M, C, C, bias=proj_b, epi='f32').view(Bp, N, C)
        ctx.save_for_backward(xh, qkv, cx, lse, qkv_wh, proj_wh)
        ctx.geom = (Bp, N, C, H)
        if probs is None:
            probs = torch.empty(0, device=x.device)
        ctx.mark_non_differentiable(probs)
        return out, probs

    @staticmethod
    def backward(ctx, dout, _dprobs):
        k = K()
        xh, qkv, cx, lse, qkv_wh, proj_wh = ctx.saved_tensors
        Bp, N, C, H = ctx.geom
        M = Bp * N
        hd = C // H
        g = k.gather_cast(dout.contiguous().view(M, C).float())
        d_proj_w = _wgrad(g, cx, C, C, M)
        d_proj_b = k.colsum(g)
        dcx = _dgrad(g, proj_wh, M, C, C, epi='bf16')
        if N <= ATTN_SINGLE_PASS_MAX:
            dqkv = k.attn_bwd(qkv, cx, dcx, lse, Bp, N, H, hd, hd ** -0.5)
        else:
            dqkv = _streaming_attn_bwd(k, qkv, cx, dcx, lse, Bp, N, H, hd)
        d_qkv_w = _wgrad(dqkv, xh, 3 * C, C, M)
        d_qkv_b = k.colsum(dqkv)
        dx = _dgrad(dqkv, qkv_wh, M, C, 3 * C, epi='f32').view(Bp, N, C)
        return dx, d_qkv_w, d_qkv_b, d_proj_w, d_proj_b, None, None, None, None


# --------------------------------------------------------------------------------------------------
class LinearSmallFn(torch.autograd.Function):
    """y = x W^T + b for a handful of rows (ClassificationHead.forward, transformer.py:78-80), fp32 GEMV kernels."""

    @staticmethod
    def forward(ctx, x, w, b):
        k = K()
        x2 = x.reshape(-1, x.shape[-1]).float().contiguous()
        y = k.linear_small_fwd(x2, w.contiguous(), b)
        ctx.save_for_backward(x2, w)
        ctx.has_bias = b is not None
        ctx.xshape = tuple(x.shape)
        return y.view(*x.shape[:-1], w.shape[0])

    @staticmethod
    def backward(ctx, dy):
        k = K()
        x2, w = ctx.saved_tensors
        dy2 = dy.reshape(-1, dy.shape[-1]).float().contiguous()
        dx, dw, db = k.linear_small_bwd(dy2, x2, w.contiguous(), need_dx=ctx.needs_input_grad[0],
                                        need_dw=ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        return (None if dx is None else dx.view(ctx.xshape)), dw, (db if ctx.has_bias else None)


class SoftmaxCEFn(torch.autograd.Function):
    """Mean softmax cross-entropy over rows: hard int64 labels (nn.CrossEntropyLoss, model_trainer.py:91) or soft fp32
    targets (timm SoftTargetCrossEntropy, :89).  Forward also produces d loss / d logits (one launch)."""

    @staticmethod
    def forward(ctx, logits, target):
        k = K()
        z = logits.float().contiguous()
        if target.dtype == torch.int64:
            loss, dz, _ = k.softmax_ce(z, labels=target)
        else:
            loss, dz, _ = k.softmax_ce(z, soft_targets=target.float())
        ctx.save_for_backward(dz)
        return loss.view(())

    @staticmethod
    def backward(ctx, dloss):
        (dz,) = ctx.saved_tensors
        return K().scale_by_scalar(dz, dloss.reshape(1).float().contiguous()), None


def cross_entropy(logits, target):
    """F.cross_entropy(logits, target) (mean reduction) / SoftTargetCrossEntropy()(logits, target) on the repo's kernel."""
    return SoftmaxCEFn.apply(logits, target)
