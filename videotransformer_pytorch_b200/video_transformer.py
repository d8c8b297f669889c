"""Model surface: TimeSformer and ViViT with the reference's constructor signatures, attribute names
and state-dict keys (reference video_transformer.py:20-268 and :270-557), forward/backward on the
sm_100a kernels.

Covered configurations (SURVEY.md §8a, §8f rank 4): TimeSformer `divided_space_time`, `space_only` (197-token joint
attention per frame) and `joint_space_time` (one 1569-token attention per clip, streaming tcgen05 kernel); ViViT
`fact_encoder` (model 2), `joint_space_time` (model 1) and `divided_space_time` (model 3).  Nothing falls back to eager
PyTorch.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import ops
from .mixup import MixedClip
from .transformer import PatchEmbed, TransformerContainer, get_sine_cosine_pos_emb, _f32
from .weight_init import init_from_kinetics_pretrain_, init_from_vit_pretrain_, trunc_normal_


def _load_pretrained(module, **vit_kwargs):
    """reference video_transformer.py:154-165 / :434-451: image (ViT) or kinetics checkpoint by `weights_from`."""
    if module.pretrain_pth is None:
        return
    if module.weights_from == 'imagenet':
        init_from_vit_pretrain_(module, module.pretrain_pth, module.conv_type, module.attention_type, module.copy_strategy,
                                **vit_kwargs)
    elif module.weights_from == 'kinetics':
        init_from_kinetics_pretrain_(module, module.pretrain_pth)
    else:
        raise TypeError(f'not support the pretrained weight {module.pretrain_pth}')


class _ByteClipInput:
    """Models fed the decoder's uint8 clip [B, T, H, W, 3] (optionally wrapped in a mixup.MixedClip): ToTensor + Normalize
    (+ Mixup / CutMix) are folded into the patch-operand kernel."""

    def set_input_normalization(self, mean, std):
        """Normalisation applied when the model is fed the decoder's uint8 clip [B, T, H, W, 3] directly (the reference
        does it on the CPU: data_transform.py ToTensor + Normalize with data_trainer.py:69-73's mean / std)."""
        self._input_norm = (tuple(float(m) for m in mean), tuple(float(s) for s in std))
        self._input_norm_dev = None

    def _norm_tensors(self, device):
        cached = getattr(self, '_input_norm_dev', None)
        if cached is None or cached[0].device != device:
            mean, std = getattr(self, '_input_norm', ((0.45, 0.45, 0.45), (0.225, 0.225, 0.225)))
            scale = torch.tensor([1.0 / (255.0 * s) for s in std], dtype=torch.float32, device=device)
            shift = torch.tensor([-m / s for m, s in zip(mean, std)], dtype=torch.float32, device=device)
            cached = self._input_norm_dev = (scale, shift)
        return cached

    def _unwrap_clip(self, x):
        """-> (tensor, (scale, shift) | None, mix plan | None)"""
        plan = None
        if isinstance(x, MixedClip):
            x, plan = x.clip, x.plan
        norm = self._norm_tensors(x.device) if x.dtype == torch.uint8 else None
        if plan is not None and norm is None:
            raise RuntimeError('MixedClip must wrap a uint8 clip (float clips are mixed by Mixup.__call__ itself)')
        return x, norm, plan


class TimeSformer(_ByteClipInput, nn.Module):
    """TimeSformer (divided space-time attention).  forward(x[B,T,3,H,W]) -> [B, embed_dims]."""

    supported_attention_types = ['divided_space_time', 'space_only', 'joint_space_time']

    def __init__(self, num_frames, img_size=224, patch_size=16, pretrain_pth=None, weights_from='imagenet',
                 embed_dims=768, num_heads=12, num_transformer_layers=12, in_channels=3, conv_type='Conv2d',
                 dropout_p=0., attention_type='divided_space_time', norm_layer=nn.LayerNorm, copy_strategy='repeat',
                 use_learnable_pos_emb=True, return_cls_token=True, **kwargs):
        super().__init__()
        assert attention_type in self.supported_attention_types, f'Unsupported Attention Type {attention_type}!'
        if dropout_p:
            raise NotImplementedError('dropout_p > 0 is not on the reference hot path (always 0.)')
        self.num_frames = num_frames
        self.pretrain_pth = pretrain_pth
        self.weights_from = weights_from
        self.embed_dims = embed_dims
        self.num_transformer_layers = num_transformer_layers
        self.attention_type = attention_type
        self.copy_strategy = copy_strategy
        self.conv_type = conv_type
        self.use_learnable_pos_emb = use_learnable_pos_emb
        self.return_cls_token = return_cls_token

        self.patch_embed = PatchEmbed(img_size=img_size, patch_size=patch_size, in_channels=in_channels,
                                      embed_dims=embed_dims, conv_type=conv_type)
        num_patches = self.patch_embed.num_patches
        operator_order = ['time_attn', 'space_attn', 'ffn'] if attention_type == 'divided_space_time' else ['self_attn', 'ffn']
        self.transformer_layers = TransformerContainer(
            num_transformer_layers=num_transformer_layers, embed_dims=embed_dims, num_heads=num_heads,
            num_frames=num_frames, norm_layer=norm_layer, hidden_channels=embed_dims * 4,
            operator_order=operator_order)
        self.norm = norm_layer(embed_dims, eps=1e-6)

        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dims))
        self.use_cls_token_temporal = operator_order[-2] == 'time_attn'     # False: cls lives in pos_embed
        num_patches = num_patches + 1
        if use_learnable_pos_emb:
            self.pos_embed = nn.Parameter(torch.zeros(1, num_patches, embed_dims))
        else:
            self.pos_embed = get_sine_cosine_pos_emb(num_patches, embed_dims)
        self.drop_after_pos = nn.Dropout(p=dropout_p)
        if attention_type != 'space_only':          # space_only has no temporal embedding (reference :137-142)
            if use_learnable_pos_emb:
                self.time_embed = nn.Parameter(torch.zeros(1, num_frames, embed_dims))
            else:
                self.time_embed = get_sine_cosine_pos_emb(num_frames, embed_dims)
            self.drop_after_time = nn.Dropout(p=dropout_p)
        self.init_weights()

    def init_weights(self):
        if self.use_learnable_pos_emb:
            nn.init.trunc_normal_(self.pos_embed, std=.02)
            if self.attention_type != 'space_only':
                nn.init.trunc_normal_(self.time_embed, std=.02)
        trunc_normal_(self.cls_token, std=.02)
        _load_pretrained(self)

    @torch.jit.ignore
    def no_weight_decay_keywords(self):
        return {'pos_embed', 'cls_token', 'mask_token'}

    def interpolate_pos_encoding(self, x, w, h):
        """reference video_transformer.py:171-191: the spatial position table for tokens `x` ([*, 1 + npatch, D], cls
        first) of a clip of width w and height h — pos_embed itself when the grid is the model's own, else its patch rows
        resampled bicubically (F.interpolate with scale factors (w//p + 0.1) / sqrt(N), (h//p + 0.1) / sqrt(N)) on the
        device.  As in the reference the result has w//p rows and h//p columns, flattened row-major: for w != h it is
        added to tokens in (h//p, w//p) raster order, i.e. transposed.  Reproduced, not fixed."""
        pos = self.pos_embed if self.use_learnable_pos_emb else self.pos_embed.to(x.device).detach()
        return self._resampled_pos(pos, x.shape[1] - 1, w, h)

    def _resampled_pos(self, pos, npatch, w, h):
        N = pos.shape[1] - 1
        if npatch == N and w == h:
            return pos
        gh, gw = (s // p for s, p in zip(self.patch_embed.img_size, self.patch_embed.patch_size))
        if gh != gw:
            raise NotImplementedError(f'pos_embed interpolation needs a square patch grid; this model has {gh} x {gw} '
                                      f'patches (img_size {self.patch_embed.img_size}), so it only takes clips of that size')
        p = self.patch_embed.patch_size[0]
        sq = math.sqrt(N)
        sf_r, sf_c = (w // p + 0.1) / sq, (h // p + 0.1) / sq          # the `+ 0.1` of the reference (:183)
        rows, cols = math.floor(gh * sf_r), math.floor(gh * sf_c)      # F.interpolate's output size for a scale factor
        assert (rows, cols) == (w // p, h // p), (rows, cols, w, h)
        # ATen samples at (dst + 0.5) / scale_factor - 0.5 with 1 / scale_factor taken in double, then cast to float
        return ops.PosEmbedInterpFn.apply(pos, gh, rows, cols, 1.0 / sf_r, 1.0 / sf_c)

    def _embeds(self, x):
        pos = self.pos_embed
        tim = self.time_embed if self.attention_type != 'space_only' else None
        if not self.use_learnable_pos_emb:
            pos = pos.to(x.device).detach()
            tim = None if tim is None else tim.to(x.device).detach()
        return pos, tim

    def prepare_tokens(self, x):
        x, norm, plan = self._unwrap_clip(x)
        if norm is not None:                # [B, T, H, W, C] bytes
            b, t, h, w, c = x.shape
        else:
            b, t, c, h, w = x.shape
        pe = self.patch_embed
        ph, pw = pe.projection.kernel_size
        if h % ph or w % pw or pw % 8:
            raise NotImplementedError(f'input {h} x {w}: the patch kernels need H % {ph} == 0, W % {pw} == 0 and a patch '
                                      f'width that is a multiple of 8 (patch {ph} x {pw})')
        pos, tim = self._embeds(x)
        pos = self._resampled_pos(pos, (h // ph) * (w // pw), w, h)
        mode = 'frames' if self.attention_type == 'space_only' else 'timesformer'   # space_only: per-frame tokens
        tok = ops.PatchTokensFn.apply(x, _f32(pe.projection.weight), _f32(pe.projection.bias), self.cls_token, pos, tim,
                                      pe.shadow(), mode, 1, norm, plan)
        return tok, b

    def forward(self, x):
        x, b = self.prepare_tokens(x)
        x = self.transformer_layers(x)
        if self.attention_type == 'space_only':      # '(b t) p d -> b p d' mean over frames (reference :247-249)
            x = x.view(b, x.shape[0] // b, x.shape[1], x.shape[2]).mean(dim=1)
        S = x.shape[1]
        if self.return_cls_token:
            if self.attention_type == 'space_only':
                rows = (torch.arange(b, device=x.device, dtype=torch.int32) * S).contiguous()
                return ops.RowsNormFn.apply(x, _f32(self.norm.weight), _f32(self.norm.bias), self.norm.eps, rows)
            rows = ops.token_maps(b, self.num_frames, (S - 1) // self.num_frames, str(x.device))['cls_rows']
            return ops.RowsNormFn.apply(x, _f32(self.norm.weight), _f32(self.norm.bias), self.norm.eps, rows)
        y = ops.RowsNormFn.apply(x, _f32(self.norm.weight), _f32(self.norm.bias), self.norm.eps, None)
        return y.view(b, S, -1)[:, 1:].mean(1)

    def get_last_selfattention(self, x):
        x, b = self.prepare_tokens(x)
        return self.transformer_layers(x, return_attention=True)


def get_vit_base_patch16_224(**kwargs):
    return TimeSformer(num_frames=kwargs['num_frames'], pretrain_pth=kwargs['pretrain_pth'],
                       weights_from=kwargs['weights_from'], img_size=kwargs['img_size'],
                       attention_type=kwargs['attention_type'], patch_size=16, embed_dims=768, num_heads=12,
                       in_channels=3, num_transformer_layers=12, conv_type='Conv2d', dropout_p=0.,
                       norm_layer=nn.LayerNorm, copy_strategy='repeat', use_learnable_pos_emb=True,
                       return_cls_token=True)


class ViViT(_ByteClipInput, nn.Module):
    """ViViT factorised encoder (model 2): tubelet embed -> 12 spatial layers per frame ->
    frame tokens (+ the reference's `x[:b,0,:]` cls gather) -> 4 temporal layers."""

    supported_attention_types = ['fact_encoder', 'joint_space_time', 'divided_space_time']

    def __init__(self, num_frames, img_size=224, patch_size=16, pretrain_pth=None, weights_from='imagenet',
                 embed_dims=768, num_heads=12, num_transformer_layers=12, in_channels=3, dropout_p=0., tube_size=2,
                 conv_type='Conv3d', attention_type='fact_encoder', norm_layer=nn.LayerNorm, copy_strategy='repeat',
                 extend_strategy='temporal_avg', use_learnable_pos_emb=True, return_cls_token=True, **kwargs):
        super().__init__()
        assert attention_type in self.supported_attention_types, f'Unsupported Attention Type {attention_type}!'
        if dropout_p:
            raise NotImplementedError('dropout_p > 0 is not on the reference hot path (always 0.)')
        if conv_type != 'Conv3d':
            raise NotImplementedError('ViViT hot path uses the Conv3d tubelet embedding')
        num_frames = num_frames // tube_size
        self.num_frames = num_frames
        self.pretrain_pth = pretrain_pth
        self.weights_from = weights_from
        self.embed_dims = embed_dims
        self.num_transformer_layers = num_transformer_layers
        self.attention_type = attention_type
        self.conv_type = conv_type
        self.copy_strategy = copy_strategy
        self.extend_strategy = extend_strategy
        self.tube_size = tube_size
        self.num_time_transformer_layers = 4 if attention_type == 'fact_encoder' else 0
        self.use_learnable_pos_emb = use_learnable_pos_emb
        self.return_cls_token = return_cls_token

        self.patch_embed = PatchEmbed(img_size=img_size, patch_size=patch_size, in_channels=in_channels,
                                      embed_dims=embed_dims, tube_size=tube_size, conv_type=conv_type)
        num_patches = self.patch_embed.num_patches
        mk = lambda n, order: TransformerContainer(
            num_transformer_layers=n, embed_dims=embed_dims, num_heads=num_heads, num_frames=num_frames,
            norm_layer=norm_layer, hidden_channels=embed_dims * 4, operator_order=order)
        if attention_type == 'divided_space_time':          # model 3 (reference :349-360)
            self.transformer_layers = mk(num_transformer_layers, ['time_attn', 'space_attn', 'ffn'])
        elif attention_type == 'joint_space_time':          # model 1 (:361-373): one 1+P*T' token attention per clip
            self.transformer_layers = mk(num_transformer_layers, ['self_attn', 'ffn'])
        else:                                               # model 2, factorised encoder (:374-400)
            self.transformer_layers = nn.ModuleList([mk(num_transformer_layers, ['self_attn', 'ffn']),
                                                     mk(self.num_time_transformer_layers, ['self_attn', 'ffn'])])
        self.norm = norm_layer(embed_dims, eps=1e-6)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dims))
        # reference :405-416: only fact_encoder has a cls slot in time_embed; operator_order[-2] is never 'time_attn'
        self.use_cls_token_temporal = False
        n_time = num_frames + 1 if attention_type == 'fact_encoder' else num_frames
        if use_learnable_pos_emb:
            self.pos_embed = nn.Parameter(torch.zeros(1, num_patches + 1, embed_dims))
            self.time_embed = nn.Parameter(torch.zeros(1, n_time, embed_dims))
        else:
            self.pos_embed = get_sine_cosine_pos_emb(num_patches + 1, embed_dims)
            self.time_embed = get_sine_cosine_pos_emb(n_time, embed_dims)
        self.drop_after_pos = nn.Dropout(p=dropout_p)
        self.drop_after_time = nn.Dropout(p=dropout_p)
        self.init_weights()

    def init_weights(self):
        if self.use_learnable_pos_emb:
            nn.init.trunc_normal_(self.pos_embed, std=.02)
            nn.init.trunc_normal_(self.time_embed, std=.02)
        trunc_normal_(self.cls_token, std=.02)
        _load_pretrained(self, extend_strategy=self.extend_strategy, tube_size=self.tube_size,
                         num_time_transformer_layers=self.num_time_transformer_layers)

    @torch.jit.ignore
    def no_weight_decay_keywords(self):
        return {'pos_embed', 'cls_token', 'mask_token'}

    def prepare_tokens(self, x):
        x, norm, plan = self._unwrap_clip(x)
        b = x.shape[0]
        h, w = x.shape[2:4] if norm is not None else x.shape[3:5]
        pe = self.patch_embed
        if (h // pe.patch_size[0]) * (w // pe.patch_size[1]) != pe.num_patches:
            raise NotImplementedError(f'ViViT takes clips of img_size {pe.img_size} only (got {h} x {w}): like the reference '
                                      f'it adds pos_embed without interpolation')
        pos = self.pos_embed if self.use_learnable_pos_emb else self.pos_embed.to(x.device).detach()
        if self.attention_type == 'fact_encoder':
            tok = ops.PatchTokensFn.apply(x, _f32(pe.projection.weight), _f32(pe.projection.bias), self.cls_token, pos, None,
                                          pe.shadow(), 'frames', self.tube_size, norm, plan)
        else:
            # reference :476-499 with use_cls_token_temporal False == TimeSformer's assembly on tubelets: one cls,
            # tokens 'b (p t) d', pos_embed per patch + time_embed per tubelet (fused into the patch GEMM epilogue)
            tim = self.time_embed if self.use_learnable_pos_emb else self.time_embed.to(x.device).detach()
            tok = ops.PatchTokensFn.apply(x, _f32(pe.projection.weight), _f32(pe.projection.bias), self.cls_token, pos, tim,
                                          pe.shadow(), 'timesformer', self.tube_size, norm, plan)
        cls_tokens = self.cls_token.expand(tok.shape[0], -1, -1)
        return tok, cls_tokens, b

    def _temporal_tokens(self, x, b):
        # reference video_transformer.py:515-523.  NOTE the quirk at :515: `x[:b, 0, :]` indexes the
        # (b t)-major tensor, i.e. it takes the cls of sample 0 / frames 0..b-1 — reproduced, not fixed.
        cls_tokens = x[:b, 0, :].unsqueeze(1)
        tim = self.time_embed if self.use_learnable_pos_emb else self.time_embed.to(x.device).detach()
        frames = x[:, 1:, :].reshape(b, x.shape[0] // b, x.shape[1] - 1, x.shape[2]).mean(dim=2)
        return torch.cat((cls_tokens, frames), dim=1) + tim

    def forward(self, x):
        x, cls_tokens, b = self.prepare_tokens(x)
        if self.attention_type != 'fact_encoder':
            x = self.transformer_layers(x)
        else:
            spatial, temporal = self.transformer_layers
            x = spatial(x)
            x = self._temporal_tokens(x, b)
            x = temporal(x)
        if self.return_cls_token:
            S = x.shape[1]
            rows = (torch.arange(b, device=x.device, dtype=torch.int32) * S).contiguous()
            return ops.RowsNormFn.apply(x, _f32(self.norm.weight), _f32(self.norm.bias), self.norm.eps, rows)
        y = ops.RowsNormFn.apply(x, _f32(self.norm.weight), _f32(self.norm.bias), self.norm.eps, None)
        return y.view(x.shape)[:, 1:].mean(1)

    def get_last_selfattention(self, x):
        x, cls_tokens, b = self.prepare_tokens(x)
        if self.attention_type != 'fact_encoder':
            return self.transformer_layers(x, return_attention=True)
        spatial, temporal = self.transformer_layers
        x = spatial(x)
        x = self._temporal_tokens(x, b)
        return temporal(x, return_attention=True)
