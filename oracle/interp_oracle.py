"""Plain-torch CPU restatement of TimeSformer fed clips of another size than img_size.

TEST INFRASTRUCTURE (see oracle/__init__.py).  It extends ``vt_oracle`` (whose blocks and primitives it reuses) with
``TimeSformer.interpolate_pos_encoding`` (reference video_transformer.py:171-191) in ``prepare_tokens`` (:193-240), for
the three attention types.  At the model's own size the interpolation is the identity and every function computes what
the matching ``vt_oracle`` function computes.

Pinned against the real reference class by ``oracle/make_golden_interp.py``; the fixtures it writes
(``tests/golden/timesformer_interp_*.npz``) hold the clip and the parameters as seeds plus the key / shape list, and are
read back with ``load_golden``.
"""
from __future__ import annotations

import json
import math
import os
import types

import numpy as np
import torch

from oracle import vt_oracle as O

ORDER = {'divided_space_time': ['time_attn', 'space_attn', 'ffn'], 'space_only': ['self_attn', 'ffn'],
         'joint_space_time': ['self_attn', 'ffn']}


def interpolate_pos_encoding(pos_embed, npatch, w, h, patch):
    """TimeSformer.interpolate_pos_encoding, video_transformer.py:171-191, with the same F.interpolate call: for another
    patch count or a non-square clip the S x S patch table is resampled bicubically with scale factors
    (w//p + 0.1) / S, (h//p + 0.1) / S to w//p rows and h//p columns and flattened row-major (transposed w.r.t. the
    (h//p, w//p) token raster when w != h — the reference's behaviour)."""
    N = pos_embed.shape[1] - 1
    if npatch == N and w == h:                                            # :174-175
        return pos_embed
    D = pos_embed.shape[-1]
    w0, h0 = w // patch + 0.1, h // patch + 0.1                           # :179-183
    grid = pos_embed[:, 1:].reshape(1, int(math.sqrt(N)), int(math.sqrt(N)), D).permute(0, 3, 1, 2)
    grid = torch.nn.functional.interpolate(grid, scale_factor=(w0 / math.sqrt(N), h0 / math.sqrt(N)), mode='bicubic')
    assert int(w0) == grid.shape[-2] and int(h0) == grid.shape[-1]         # :189
    return torch.cat((pos_embed[:, :1], grid.permute(0, 2, 3, 1).reshape(1, -1, D)), dim=1)


def tokens(sd, x, cfg, attention_type):
    """TimeSformer.prepare_tokens, video_transformer.py:193-240: [B, 1 + P*T, D] ('b (p t) d', one cls), or per-frame
    [(b t), 1 + P, D] for space_only (no time embedding)."""
    B = x.shape[0]
    tok = O.patch_embed(x, sd['patch_embed.projection.weight'], sd['patch_embed.projection.bias'])
    BT, P, D = tok.shape
    pos = interpolate_pos_encoding(sd['pos_embed'], P, x.shape[-1], x.shape[-2], sd['patch_embed.projection.weight'].shape[-2])
    tok = torch.cat((sd['cls_token'].expand(BT, 1, D), tok), dim=1) + pos   # :207-209
    if attention_type == 'space_only':
        return tok
    T = BT // B
    cls_tokens = tok[:B, 0, :].unsqueeze(1)                               # :216
    tok = tok[:, 1:, :].reshape(B, T, P, D).permute(0, 2, 1, 3).reshape(B * P, T, D) + sd['time_embed']   # :231-233
    return torch.cat((cls_tokens, tok.reshape(B, P * T, D)), dim=1)      # :236-237


def forward(sd, x, cfg, attention_type, training=False):
    """TimeSformer.forward, video_transformer.py:242-256."""
    tok = tokens(sd, x, cfg, attention_type)
    tok = O.container(tok, sd, 'transformer_layers.', cfg['num_transformer_layers'], ORDER[attention_type],
                      cfg['num_frames'], cfg['num_heads'], training)
    if attention_type == 'space_only':                                    # :247-249
        B, T = x.shape[0], x.shape[1]
        tok = tok.reshape(B, T, tok.shape[1], tok.shape[2]).mean(dim=1)
    tok = O.layer_norm(tok, sd['norm.weight'], sd['norm.bias'], 1e-6)
    return tok[:, 0]


def last_selfattention(sd, x, cfg, attention_type):
    """TimeSformer.get_last_selfattention, video_transformer.py:258-261."""
    return O.container(tokens(sd, x, cfg, attention_type), sd, 'transformer_layers.', cfg['num_transformer_layers'],
                       ORDER[attention_type], cfg['num_frames'], cfg['num_heads'], False, return_attention=True)


# ----------------------------------------------------------------------------
# seeded parameters and clips (the fixtures store seeds, not values)
# ----------------------------------------------------------------------------
def seeded_state(named_shapes, seed):
    """Reference-format state dict with every tensor drawn from one seeded generator in the given key order; values are
    fp32-representable (returned as fp64).  Norm weights 1 + N(0, 0.1), biases N(0, 0.05), the position / time tables
    N(0, 0.5) (large enough that a wrong resampling shows in every output), cls N(0, 0.02), weights N(0, 1/fan_in)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name, shape in named_shapes:
        r = torch.randn(tuple(shape), generator=g, dtype=torch.float64)
        if name.endswith('norm.weight'):
            v = 1.0 + 0.1 * r
        elif name.endswith('bias'):
            v = 0.05 * r
        elif name in ('pos_embed', 'time_embed'):
            v = 0.5 * r
        elif name == 'cls_token':
            v = 0.02 * r
        else:
            v = r / math.sqrt(int(np.prod(shape[1:])))
        sd[name] = v.float().double()
    return sd


def seeded_clip(shape, seed):
    return torch.randn(tuple(shape), generator=torch.Generator().manual_seed(seed), dtype=torch.float64).float().double()


def load_golden(name, gold_dir):
    """A fixture of make_golden_interp.py: x / sd regenerated from their seeds (fp32), reference outputs (fp64),
    gradients verbatim (small) or as [sum, l2, <g, linspace(-1,1)>] checksums, cfg, attention type, DropPath seed."""
    z = np.load(os.path.join(gold_dir, name + '.npz'))
    named_shapes = json.loads(str(z['named_shapes']))
    g = types.SimpleNamespace()
    g.attention_type = str(z['attention_type'])
    g.cfg = {k[4:]: int(z[k]) for k in z.files if k.startswith('cfg_')}
    g.sd = {k: v.float() for k, v in seeded_state(named_shapes, int(z['param_seed'])).items()}
    g.x = seeded_clip(z['x_shape'].tolist(), int(z['x_seed'])).float()
    g.out = {k[5:]: torch.from_numpy(z[k]) for k in z.files if k.startswith('out::')}
    y = g.out['y_train']                                                  # the train-mode loss is sum(y * loss_w)
    g.out['loss_w'] = torch.linspace(-1, 1, y.numel(), dtype=torch.float64).reshape(y.shape)
    g.grad = {k[6:]: torch.from_numpy(z[k]) for k in z.files if k.startswith('grad::')}
    g.gradsum = {k[9:]: z[k] for k in z.files if k.startswith('gradsum::')}
    g.train_seed = int(z['train_seed'])
    return g
