"""Golden vectors of TimeSformer fed clips of another size than img_size, from the REAL reference class.

Run where the reference checkout exists (like oracle/make_golden.py, whose reference import it uses):

    python oracle/make_golden_interp.py [name ...]

For each case the reference TimeSformer (video_transformer.py:20-261, interpolate_pos_encoding :171-191 live in
prepare_tokens) is run in fp64 on seeded parameters and a seeded clip; oracle/interp_oracle.py must agree to 1e-12 on
the eval output, tokens and last-layer attention, and on the train-mode output (seeded DropPath), dx and every parameter
gradient.  The .npz holds seeds and the key / shape list instead of parameter and clip values, the reference outputs,
dx, and the gradients (small ones verbatim, large ones as checksums); interp_oracle.load_golden reads it back.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.make_golden import GOLD, import_reference, pack_grads, rel  # noqa: E402

CASES = [   # (name, attention type, model img_size, input (H, W)); head dim 64 as the GPU attention kernels need
    ('timesformer_interp_up', 'divided_space_time', 32, (64, 64)),
    ('timesformer_interp_down', 'divided_space_time', 64, (32, 32)),
    ('timesformer_interp_nonsquare', 'divided_space_time', 32, (32, 64)),
    ('timesformer_interp_space_only', 'space_only', 32, (64, 64)),
    ('timesformer_interp_joint', 'joint_space_time', 32, (64, 64)),
]


def interp_case(vt, name, cfg, B, seed, attention_type, hw):
    from oracle import interp_oracle as IO
    m = vt.TimeSformer(num_frames=cfg['num_frames'], img_size=cfg['img_size'], patch_size=cfg['patch_size'],
                       embed_dims=cfg['embed_dims'], num_heads=cfg['num_heads'],
                       num_transformer_layers=cfg['num_transformer_layers'], attention_type=attention_type).double()
    named_shapes = [(k, list(v.shape)) for k, v in m.state_dict().items()]
    sd = IO.seeded_state(named_shapes, seed)
    m.load_state_dict(sd, strict=True)
    x_shape = (B, cfg['num_frames'], 3, hw[0], hw[1])
    x = IO.seeded_clip(x_shape, seed + 1)
    m.eval()
    with torch.no_grad():
        y_eval = m(x)
        tok = m.prepare_tokens(x)[0]
        attn = m.get_last_selfattention(x)
        assert rel(IO.forward(sd, x, cfg, attention_type), y_eval) < 1e-12
        assert rel(IO.tokens(sd, x, cfg, attention_type), tok) < 1e-12
        assert rel(IO.last_selfattention(sd, x, cfg, attention_type), attn) < 1e-12
    m.train()
    xg = x.clone().requires_grad_(True)
    torch.manual_seed(5000 + seed)
    y_tr = m(xg)
    w = torch.linspace(-1, 1, y_tr.numel(), dtype=torch.float64).reshape(y_tr.shape)
    (y_tr * w).sum().backward()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xo = x.clone().requires_grad_(True)
    torch.manual_seed(5000 + seed)
    yo = IO.forward(sdg, xo, cfg, attention_type, training=True)
    (yo * w).sum().backward()
    assert rel(yo.detach(), y_tr.detach()) < 1e-12
    assert rel(xo.grad, xg.grad) < 1e-10
    for n, g in grads.items():
        assert rel(sdg[n].grad, g) < 1e-9, n
    print(f'[{name}] oracle == reference ({attention_type}, {cfg["img_size"]}^2 model fed {hw[0]}x{hw[1]}: eval, tokens, '
          f'last_attn, train fwd, dx, all {len(grads)} grads)')
    save = {'x_seed': np.int64(seed + 1), 'x_shape': np.asarray(x_shape, dtype=np.int64), 'param_seed': np.int64(seed),
            'named_shapes': np.array(json.dumps(named_shapes)), 'attention_type': np.array(attention_type),
            'train_seed': np.int64(5000 + seed), 'B': np.int64(B)}
    for k, v in cfg.items():
        save['cfg_' + k] = np.int64(v)
    save['out::y_eval'] = y_eval.numpy()
    save['out::tokens'] = tok.numpy()
    save['out::last_attn'] = attn.numpy()
    save['out::y_train'] = y_tr.detach().numpy()
    save['out::dx'] = xg.grad.float().numpy()
    pack_grads(save, grads)
    np.savez_compressed(os.path.join(GOLD, name + '.npz'), **save)


def main():
    _, vt, _ = import_reference()
    only = set(sys.argv[1:])
    for i, (name, attention_type, img, hw) in enumerate(CASES):
        if not only or name in only:
            cfg = dict(num_frames=2, img_size=img, patch_size=16, embed_dims=128, num_heads=2, num_transformer_layers=2)
            interp_case(vt, name, cfg, B=2, seed=20 + i, attention_type=attention_type, hw=hw)


if __name__ == '__main__':
    main()
