"""pretrain_pth checkpoint loaders (weight_init.py) against the reference's own functions (weight_init.py:107-314).

The remapped state dicts of synthetic checkpoints are compared key by key and bit for bit with what the reference loaders
produced from the same checkpoints (tests/golden/checkpoint_remaps.json, written by `oracle/make_golden.py
checkpoint_remaps`).  The constructors' `pretrain_pth` flow is exercised with a synthetic checkpoint as well: the drop-in
claim must hold for the reference's standard finetune flow."""
import hashlib
import json
import os

import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'checkpoint_remaps.json')
REMAP_CASES = [
    ('Conv2d', 'divided_space_time', 'repeat', 'temporal_avg'), ('Conv2d', 'space_only', 'repeat', 'temporal_avg'),
    ('Conv3d', 'fact_encoder', 'repeat', 'temporal_avg'), ('Conv3d', 'fact_encoder', 'set_zero', 'center_frame'),
    ('Conv3d', 'joint_space_time', 'repeat', 'center_frame'), ('Conv2d', 'divided_space_time', 'set_zero', 'temporal_avg')]


def remap_case_id(kind, *case):
    return '/'.join((kind,) + case)


def state_digest(sd):
    """key -> [dtype, shape, SHA-256 prefix of the contiguous tensor bytes]"""
    return {k: [str(v.dtype), list(v.shape), hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest()[:16]]
            for k, v in sd.items()}


@pytest.fixture(scope='module')
def reference_remaps():
    with open(GOLDEN) as fh:
        return json.load(fh)


def _vit_image_checkpoint(D=32, L=2, P=4):
    """Keys of an mmaction-style ViT image checkpoint as init_from_vit_pretrain_ expects them."""
    g = torch.Generator().manual_seed(0)
    rn = lambda *s: torch.randn(*s, generator=g)
    sd = {'cls_token': rn(1, 1, D), 'pos_embed': rn(1, P + 1, D), 'patch_embed.projection.weight': rn(D, 3, 16, 16),
          'patch_embed.projection.bias': rn(D), 'norm.weight': rn(D), 'norm.bias': rn(D)}
    for i in range(L):
        p = f'transformer_layers.layers.{i}.'
        sd[p + 'attentions.0.attn.in_proj_weight'] = rn(3 * D, D)
        sd[p + 'attentions.0.attn.in_proj_bias'] = rn(3 * D)
        sd[p + 'attentions.0.attn.out_proj.weight'] = rn(D, D)
        sd[p + 'attentions.0.attn.out_proj.bias'] = rn(D)
        sd[p + 'norms.0.weight'], sd[p + 'norms.0.bias'] = rn(D), rn(D)
        sd[p + 'norms.1.weight'], sd[p + 'norms.1.bias'] = rn(D), rn(D)
        sd[p + 'ffns.0.layers.0.0.weight'], sd[p + 'ffns.0.layers.0.0.bias'] = rn(4 * D, D), rn(4 * D)
        sd[p + 'ffns.0.layers.1.weight'], sd[p + 'ffns.0.layers.1.bias'] = rn(D, 4 * D), rn(D)
    return sd


def _mae_checkpoint(D=32, L=2):
    g = torch.Generator().manual_seed(1)
    rn = lambda *s: torch.randn(*s, generator=g)
    sd = {'encoder.patch_embed.proj.weight': rn(D, 3, 16, 16), 'encoder.patch_embed.proj.bias': rn(D),
          'encoder.norm.weight': rn(D), 'encoder.norm.bias': rn(D), 'decoder.blocks.0.foo': rn(3)}
    for i in range(L):
        p = f'encoder.blocks.{i}.'
        sd[p + 'norm1.weight'], sd[p + 'norm1.bias'] = rn(D), rn(D)
        sd[p + 'norm2.weight'], sd[p + 'norm2.bias'] = rn(D), rn(D)
        sd[p + 'attn.q_bias'], sd[p + 'attn.v_bias'] = rn(D), rn(D)
        sd[p + 'attn.qkv.weight'], sd[p + 'attn.proj.weight'], sd[p + 'attn.proj.bias'] = rn(3 * D, D), rn(D, D), rn(D)
        sd[p + 'mlp.fc1.weight'], sd[p + 'mlp.fc1.bias'] = rn(4 * D, D), rn(4 * D)
        sd[p + 'mlp.fc2.weight'], sd[p + 'mlp.fc2.bias'] = rn(D, 4 * D), rn(D)
    return sd


def _kinetics_checkpoint():
    g = torch.Generator().manual_seed(2)
    return {'model.cls_token': torch.randn(1, 1, 8, generator=g), 'model.a.attn.in_proj_weight': torch.randn(24, 8, generator=g),
            'model.a.attn.out_proj.bias': torch.randn(8, generator=g), 'cls_head.cls_head.weight': torch.randn(4, 8, generator=g)}


@pytest.mark.parametrize('conv_type,attention_type,copy_strategy,extend', REMAP_CASES)
def test_vit_and_mae_remaps_equal_the_reference(reference_remaps, conv_type, attention_type, copy_strategy, extend):
    from videotransformer_pytorch_b200 import weight_init as W
    for kind, make, mine in (('vit', _vit_image_checkpoint, W.remap_vit_checkpoint),
                             ('mae', _mae_checkpoint, W.remap_mae_checkpoint)):
        theirs = reference_remaps[remap_case_id(kind, conv_type, attention_type, copy_strategy, extend)]
        got = state_digest(mine(make(), conv_type, attention_type, copy_strategy, extend, 2, 1))
        assert sorted(got.keys()) == sorted(theirs.keys()), kind
        for k in got:
            assert got[k] == theirs[k], (kind, k)


def test_kinetics_remap_equals_the_reference(reference_remaps):
    from videotransformer_pytorch_b200 import weight_init as W
    mine = state_digest(W.remap_kinetics_checkpoint(_kinetics_checkpoint()))
    assert mine == reference_remaps['kinetics']


def test_constructors_accept_pretrain_pth(tmp_path):
    """TimeSformer / ViViT(pretrain_pth=...) as model_trainer.py:57-74 calls them: an image checkpoint initialises both
    attentions of a divided block and the first temporal layers of the factorised encoder."""
    from videotransformer_pytorch_b200 import TimeSformer, ViViT
    ck = _vit_image_checkpoint(D=32, L=2, P=4)
    path = str(tmp_path / 'vit.pth')
    torch.save({'state_dict': ck}, path)
    kw = dict(img_size=32, patch_size=16, embed_dims=32, num_heads=4, num_transformer_layers=2)
    m = TimeSformer(num_frames=4, pretrain_pth=path, weights_from='imagenet', **kw)
    sd = m.state_dict()
    w = ck['transformer_layers.layers.1.attentions.0.attn.in_proj_weight']
    assert torch.equal(sd['transformer_layers.layers.1.attentions.0.attn.qkv.weight'], w)
    assert torch.equal(sd['transformer_layers.layers.1.attentions.1.attn.qkv.weight'], w)       # copy_strategy='repeat'
    assert torch.equal(sd['transformer_layers.layers.0.ffns.0.norm.weight'], ck['transformer_layers.layers.0.norms.1.weight'])
    assert torch.equal(sd['pos_embed'], ck['pos_embed'])
    v = ViViT(num_frames=8, pretrain_pth=path, weights_from='imagenet', **kw)
    sv = v.state_dict()
    assert torch.equal(sv['patch_embed.projection.weight'][:, :, 0], ck['patch_embed.projection.weight'] / 2)   # temporal_avg
    assert torch.equal(sv['transformer_layers.0.layers.1.attentions.0.attn.proj.weight'],
                       ck['transformer_layers.layers.1.attentions.0.attn.out_proj.weight'])
    assert torch.equal(sv['transformer_layers.1.layers.1.attentions.0.attn.proj.weight'],
                       ck['transformer_layers.layers.1.attentions.0.attn.out_proj.weight'])
    with pytest.raises(TypeError):
        TimeSformer(num_frames=4, pretrain_pth=path, weights_from='somewhere', **kw)
    # kinetics flow: a Lightning checkpoint of the trainer (model.* / cls_head.* prefixes)
    lk = {'model.' + k: val for k, val in m.state_dict().items()}
    lk['cls_head.cls_head.weight'] = torch.zeros(5, 32)
    kpath = str(tmp_path / 'kin.pth')
    torch.save({'state_dict': lk}, kpath)
    m2 = TimeSformer(num_frames=4, pretrain_pth=kpath, weights_from='kinetics', **kw)
    for k, val in m.state_dict().items():
        assert torch.equal(m2.state_dict()[k], val), k
