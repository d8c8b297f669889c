"""Generate the golden vectors in tests/golden from the REAL reference modules.

Run in the build container only (needs /root/reference):

    python oracle/make_golden.py

The reference is imported unmodified with `sys.modules` stubs for its
non-arithmetic top-level imports (matplotlib, pytorch_lightning.utilities.distributed,
pytorchvideo.* — SURVEY.md §8c).  For every case the script also runs the oracle
restatement (oracle/vt_oracle.py, oracle/mask_oracle.py) and asserts agreement,
i.e. this script is what pins the oracle.  Outputs are small .npz / .json files.
"""
from __future__ import annotations

import hashlib
import os
import random
import sys
import tempfile
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, 'tests', 'golden')
REF = '/root/reference'


def import_reference():
    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    stub('matplotlib'); stub('matplotlib.pyplot')
    stub('pytorch_lightning'); stub('pytorch_lightning.utilities')
    stub('pytorch_lightning.utilities.distributed', rank_zero_only=lambda f: f)
    # pytorchvideo is absent: bind its five names to the restatement so the real MaskFeat can be built
    from oracle.pytorchvideo_restated import install_stub_modules
    install_stub_modules()
    sys.path.insert(0, REF)
    import transformer, video_transformer, mask_generator  # noqa
    return transformer, video_transformer, mask_generator


def randomize(model, seed):
    """Reference init leaves temporal_fc at zero (transformer.py:228-232) and LN at
    identity; perturb everything so no branch is silently a no-op."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if 'temporal_fc' in n or n.endswith('norm.bias') or n.endswith('.bias'):
                p.add_(torch.randn(p.shape, generator=g, dtype=torch.float64).to(p.dtype) * 0.05)
            elif n.endswith('norm.weight'):
                p.add_(torch.randn(p.shape, generator=g, dtype=torch.float64).to(p.dtype) * 0.1)


def pack_grads(save, grads):
    """Small grads verbatim (fp32); large ones as 3 fp64 checksums
    [sum, l2, <g, linspace(-1,1)>] to keep fixtures small."""
    for n, g in grads.items():
        if g.numel() <= 4096:
            save['grad::' + n] = g.float().numpy()
        else:
            lin = torch.linspace(-1, 1, g.numel(), dtype=torch.float64)
            save['gradsum::' + n] = np.array([g.sum().item(), g.norm().item(),
                                              (g.reshape(-1) * lin).sum().item()])


def rel(a, b):
    return float((a - b).norm() / (b.norm() + 1e-30))


def timesformer_case(vt, name, cfg, B, seed):
    from oracle import vt_oracle as O
    torch.manual_seed(seed)
    m = vt.TimeSformer(num_frames=cfg['num_frames'], img_size=cfg['img_size'], patch_size=cfg['patch_size'],
                       embed_dims=cfg['embed_dims'], num_heads=cfg['num_heads'],
                       num_transformer_layers=cfg['num_transformer_layers'],
                       attention_type='divided_space_time')
    randomize(m, seed + 1)
    m = m.double()
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    x = torch.randn(B, cfg['num_frames'], 3, cfg['img_size'], cfg['img_size'], dtype=torch.float64)
    # fp32-representable inputs/params so fp32 consumers see identical values
    x = x.float().double()
    for k in sd:
        sd[k] = sd[k].float().double()
    m.load_state_dict(sd)

    out = {}
    m.eval()
    with torch.no_grad():
        y_eval = m(x)
        tok = m.prepare_tokens(x)[0]
        attn = m.get_last_selfattention(x)
    out['y_eval'] = y_eval
    out['tokens'] = tok
    out['last_attn'] = attn

    # train mode: DropPath live, CPU generator seeded
    m.train()
    xg = x.clone().requires_grad_(True)
    torch.manual_seed(1000 + seed)
    y_tr = m(xg)
    w = torch.linspace(-1, 1, y_tr.numel(), dtype=torch.float64).reshape(y_tr.shape)
    (y_tr * w).sum().backward()
    out['y_train'] = y_tr.detach()
    out['loss_w'] = w
    out['dx'] = xg.grad.float()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters()}

    # ---- pin the oracle ----
    with torch.no_grad():
        assert rel(O.timesformer_forward(sd, x, cfg), y_eval) < 1e-12
        assert rel(O.timesformer_tokens(sd, x, cfg), tok) < 1e-12
        assert rel(O.timesformer_last_selfattention(sd, x, cfg), attn) < 1e-12
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xo = x.clone().requires_grad_(True)
    torch.manual_seed(1000 + seed)
    yo = O.timesformer_forward(sdg, xo, cfg, training=True)
    (yo * w).sum().backward()
    assert rel(yo.detach(), y_tr.detach()) < 1e-12, rel(yo.detach(), y_tr.detach())
    assert rel(xo.grad, xg.grad) < 1e-10
    for n, g in grads.items():
        assert rel(sdg[n].grad, g) < 1e-9, (n, rel(sdg[n].grad, g))
    print(f'[{name}] oracle == reference (eval, tokens, last_attn, train fwd, all {len(grads)} grads)')

    save = {'x': x.float().numpy(), 'train_seed': np.int64(1000 + seed), 'B': np.int64(B)}
    for k, v in cfg.items():
        if isinstance(v, int):
            save['cfg_' + k] = np.int64(v)
    for k, v in sd.items():
        save['sd::' + k] = v.float().numpy()
    for k, v in out.items():
        save['out::' + k] = v.numpy()               # fp64
    pack_grads(save, grads)
    np.savez_compressed(os.path.join(GOLD, name + '.npz'), **save)


def vivit_case(vt, name, cfg, B, seed):
    from oracle import vt_oracle as O
    torch.manual_seed(seed)
    m = vt.ViViT(num_frames=cfg['num_frames_in'], img_size=cfg['img_size'], patch_size=cfg['patch_size'],
                 embed_dims=cfg['embed_dims'], num_heads=cfg['num_heads'],
                 num_transformer_layers=cfg['num_transformer_layers'], attention_type='fact_encoder')
    randomize(m, seed + 1)
    m = m.double()
    sd = {k: v.detach().clone().float().double() for k, v in m.state_dict().items()}
    m.load_state_dict(sd)
    x = torch.randn(B, cfg['num_frames_in'], 3, cfg['img_size'], cfg['img_size'], dtype=torch.float64).float().double()
    m.eval()
    with torch.no_grad():
        y_eval = m(x)
        assert rel(O.vivit_forward(sd, x, cfg), y_eval) < 1e-12
    m.train()
    xg = x.clone().requires_grad_(True)
    torch.manual_seed(2000 + seed)
    y_tr = m(xg)
    w = torch.linspace(-1, 1, y_tr.numel(), dtype=torch.float64).reshape(y_tr.shape)
    (y_tr * w).sum().backward()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xo = x.clone().requires_grad_(True)
    torch.manual_seed(2000 + seed)
    yo = O.vivit_forward(sdg, xo, cfg, training=True)
    (yo * w).sum().backward()
    assert rel(yo.detach(), y_tr.detach()) < 1e-12
    assert rel(xo.grad, xg.grad) < 1e-10
    for n, g in grads.items():
        assert rel(sdg[n].grad, g) < 1e-9, n
    print(f'[{name}] oracle == reference (eval, train fwd, all {len(grads)} grads)')
    save = {'x': x.float().numpy(), 'train_seed': np.int64(2000 + seed), 'B': np.int64(B)}
    for k, v in cfg.items():
        if isinstance(v, int):
            save['cfg_' + k] = np.int64(v)
    for k, v in sd.items():
        save['sd::' + k] = v.float().numpy()
    save['out::y_eval'] = y_eval.numpy()
    save['out::y_train'] = y_tr.detach().numpy()
    save['out::loss_w'] = w.numpy()
    save['out::dx'] = xg.grad.float().numpy()
    pack_grads(save, grads)
    np.savez_compressed(os.path.join(GOLD, name + '.npz'), **save)


def space_only_case(vt, name, cfg, B, seed, attention_type='space_only'):
    from oracle import vt_oracle as O
    oracle_fwd = O.timesformer_space_only_forward if attention_type == 'space_only' else O.timesformer_joint_forward
    torch.manual_seed(seed)
    m = vt.TimeSformer(num_frames=cfg['num_frames'], img_size=cfg['img_size'], patch_size=cfg['patch_size'],
                       embed_dims=cfg['embed_dims'], num_heads=cfg['num_heads'],
                       num_transformer_layers=cfg['num_transformer_layers'], attention_type=attention_type)
    randomize(m, seed + 1)
    m = m.double()
    sd = {k: v.detach().clone().float().double() for k, v in m.state_dict().items()}
    m.load_state_dict(sd)
    x = torch.randn(B, cfg['num_frames'], 3, cfg['img_size'], cfg['img_size'], dtype=torch.float64).float().double()
    m.eval()
    with torch.no_grad():
        y_eval = m(x)
        assert rel(oracle_fwd(sd, x, cfg), y_eval) < 1e-12
    m.train()
    torch.manual_seed(3000 + seed)
    y_tr = m(x)
    w = torch.linspace(-1, 1, y_tr.numel(), dtype=torch.float64).reshape(y_tr.shape)
    (y_tr * w).sum().backward()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    torch.manual_seed(3000 + seed)
    yo = oracle_fwd(sdg, x, cfg, training=True)
    (yo * w).sum().backward()
    assert rel(yo.detach(), y_tr.detach()) < 1e-12
    for n, g in grads.items():
        assert rel(sdg[n].grad, g) < 1e-9, n
    print(f'[{name}] oracle == reference (eval, train fwd, all {len(grads)} grads)')
    save = {'x': x.float().numpy(), 'train_seed': np.int64(3000 + seed), 'B': np.int64(B)}
    for k, v in cfg.items():
        if isinstance(v, int):
            save['cfg_' + k] = np.int64(v)
    for k, v in sd.items():
        save['sd::' + k] = v.float().numpy()
    save['out::y_eval'] = y_eval.numpy()
    save['out::y_train'] = y_tr.detach().numpy()
    save['out::loss_w'] = w.numpy()
    pack_grads(save, grads)
    np.savez_compressed(os.path.join(GOLD, name + '.npz'), **save)


def vivit_variant_case(vt, name, cfg, B, seed, attention_type):
    """ViViT 'joint_space_time' / 'divided_space_time' (video_transformer.py:349-373) vs the oracle."""
    from oracle import vt_oracle as O
    torch.manual_seed(seed)
    m = vt.ViViT(num_frames=cfg['num_frames_in'], img_size=cfg['img_size'], patch_size=cfg['patch_size'],
                 embed_dims=cfg['embed_dims'], num_heads=cfg['num_heads'],
                 num_transformer_layers=cfg['num_transformer_layers'], attention_type=attention_type)
    randomize(m, seed + 1)
    m = m.double()
    sd = {k: v.detach().clone().float().double() for k, v in m.state_dict().items()}
    m.load_state_dict(sd)
    x = torch.randn(B, cfg['num_frames_in'], 3, cfg['img_size'], cfg['img_size'], dtype=torch.float64).float().double()
    m.eval()
    with torch.no_grad():
        y_eval = m(x)
        assert rel(O.vivit_variant_forward(sd, x, cfg, attention_type), y_eval) < 1e-12
    m.train()
    torch.manual_seed(4000 + seed)
    y_tr = m(x)
    w = torch.linspace(-1, 1, y_tr.numel(), dtype=torch.float64).reshape(y_tr.shape)
    (y_tr * w).sum().backward()
    grads = {n: p.grad.detach().clone() for n, p in m.named_parameters()}
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    torch.manual_seed(4000 + seed)
    yo = O.vivit_variant_forward(sdg, x, cfg, attention_type, training=True)
    (yo * w).sum().backward()
    assert rel(yo.detach(), y_tr.detach()) < 1e-12
    for n, g in grads.items():
        assert rel(sdg[n].grad, g) < 1e-9, n
    print(f'[{name}] oracle == reference (eval, train fwd, all {len(grads)} grads)')
    save = {'x': x.float().numpy(), 'train_seed': np.int64(4000 + seed), 'B': np.int64(B)}
    for k, v in cfg.items():
        if isinstance(v, int):
            save['cfg_' + k] = np.int64(v)
    for k, v in sd.items():
        save['sd::' + k] = v.float().numpy()
    save['out::y_eval'] = y_eval.numpy()
    save['out::y_train'] = y_tr.detach().numpy()
    save['out::loss_w'] = w.numpy()
    pack_grads(save, grads)
    np.savez_compressed(os.path.join(GOLD, name + '.npz'), **save)


def mask_cases(mg):
    from oracle.mask_oracle import CubeMaskOracle
    rows = {}
    for seed in range(8):
        random.seed(seed); np.random.seed(seed)
        ref = mg.CubeMaskGenerator(input_size=(8, 14, 14), min_num_patches=16)
        masks, markers = [], []
        for _ in range(3):                       # three consecutive calls per seed
            m, mk = ref()
            masks.append(m); markers.append(mk)
        random.seed(seed); np.random.seed(seed)
        mine = CubeMaskOracle(input_size=(8, 14, 14), min_num_patches=16)
        for i in range(3):
            m2, mk2 = mine()
            assert m2.dtype == masks[i].dtype and np.array_equal(m2, masks[i]), (seed, i)
            assert mk2 == markers[i], (seed, i)
        rows[f'mask_{seed}'] = np.stack(masks).astype(np.int32)
        flat = []
        for i, mk in enumerate(markers):
            for s, n in mk:
                flat.append([i, s, n])
        rows[f'markers_{seed}'] = np.asarray(flat, dtype=np.int32)
    # SURVEY Appendix D known answers (first call)
    assert hashlib.sha256(rows['mask_0'][0].tobytes()).hexdigest()[:16] == 'c87b9c69a35b57eb'
    assert hashlib.sha256(rows['mask_1'][0].tobytes()).hexdigest()[:16] == '88bae48972b63616'
    assert hashlib.sha256(rows['mask_2'][0].tobytes()).hexdigest()[:16] == '150b214c947d31fd'
    np.savez_compressed(os.path.join(GOLD, 'cube_mask.npz'), **rows)
    print('[cube_mask] oracle == reference for seeds 0..7 x 3 calls; Appendix-D hashes ok')


def maskfeat_case(vt, name, kwargs, B, seed, with_grads=True):
    """Real ``MaskFeat`` (video_transformer.py:803-922; blocks = restated pytorchvideo) vs oracle/mvit_oracle.py."""
    from oracle import mvit_oracle as mo
    cfg = mo.maskfeat_config(**kwargs)
    ref_kwargs = dict(kwargs)
    for k in ('pool_q_stride_size', 'embed_dim_mul', 'atten_head_mul'):
        if k in ref_kwargs:
            ref_kwargs[k] = [list(r) for r in ref_kwargs[k]]
    torch.manual_seed(seed)
    model = vt.MaskFeat(**ref_kwargs).double()
    # block configuration derived by the reference factory (:707-761) == oracle's maskfeat_config
    for blk, mine in zip(model.mvit.blocks, cfg['blocks']):
        assert blk.blk == mine, (blk.blk, mine)
    assert model.embed_dims == cfg['embed_dims'] and model.downsample_rate == cfg['downsample_rate']
    sd = mo.random_maskfeat_state(cfg, seed=seed, dtype=torch.float64)
    model.load_state_dict(sd, strict=True)            # key names and shapes agree with the reference module tree
    model.train()
    g = torch.Generator().manual_seed(seed + 100)
    T, S = cfg['num_frames'], cfg['img_size']
    t, h, w = cfg['thw'][0], cfg['thw'][1] // cfg['downsample_rate'], cfg['thw'][2] // cfg['downsample_rate']
    x = torch.randn(B, T, 3, S, S, generator=g, dtype=torch.float64).float().double()   # stored as fp32
    mask = (torch.rand(B, t, h, w, generator=g) < 0.4).to(torch.float64)
    cube_marker = [[[0, 2], [t - 1, 1]] if i % 2 == 0 else [[1, t - 1]] for i in range(B)]
    target = torch.randn(B, T, h, w, cfg['feature_dim'] // cfg['stride'][0], generator=g, dtype=torch.float64).float().double()

    feats_ref = model.forward_features(x, mask)
    feats_nomask_ref = model.forward_features(x)
    pred_ref, loss_ref = model(x, target, mask.clone(), cube_marker)
    params = dict(model.named_parameters())
    grads_ref = torch.autograd.grad(loss_ref, list(params.values()), allow_unused=True)

    sdo = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    feats = mo.maskfeat_forward_features(sdo, x, mask, cfg)
    feats_nomask = mo.maskfeat_forward_features(sdo, x, None, cfg)
    pred, loss = mo.maskfeat_forward(sdo, x, target, mask, cube_marker, cfg)
    grads = torch.autograd.grad(loss, [sdo[k] for k in params], allow_unused=True)
    assert rel(feats, feats_ref) < 1e-12 and rel(feats_nomask, feats_nomask_ref) < 1e-12
    assert rel(pred, pred_ref) < 1e-12 and abs(loss.item() - loss_ref.item()) < 1e-12 * max(1, abs(loss_ref.item()))
    worst = 0.0
    for k, a, b in zip(params, grads, grads_ref):
        assert (a is None) == (b is None), k
        if a is not None:
            r = float((a - b).norm() / (b.norm() + 1e-6 * b.numel() ** 0.5))   # norm_k.bias grads are exactly 0 in theory
            if r > 1e-10:
                print('   grad mismatch', k, r, float(a.norm()), float(b.norm()))
            worst = max(worst, r)
    assert worst < 1e-10, worst
    save = dict(seed=np.int64(seed), B=np.int64(B), x=x.numpy().astype(np.float32), mask=mask.numpy().astype(np.float32),
                target=target.numpy().astype(np.float32),
                cube_marker=np.array([str(cube_marker)]),
                feats=feats_ref.detach().numpy(), feats_nomask_cls=feats_nomask_ref[:, 0].detach().numpy(),
                pred=pred_ref.detach().numpy(), loss=np.float64(loss_ref.item()),
                cfg_kwargs=np.array([repr(kwargs)]))
    if with_grads:
        # norm_k.bias shifts every score of a query equally => its gradient is 0 up to rounding noise: not stored
        pack_grads(save, {k: gr for k, gr in zip(params, grads_ref)
                          if gr is not None and not k.endswith('attn.norm_k.bias')})
    np.savez_compressed(os.path.join(GOLD, name + '.npz'), **save)
    print(f'[{name}] oracle == reference MaskFeat: feats/pred/loss < 1e-12, worst grad rel {worst:.2e}; '
          f'loss {loss_ref.item():.6f}')


def main():
    os.makedirs(GOLD, exist_ok=True)
    tr, vt, mg = import_reference()
    only = set(sys.argv[1:])          # optional: names of the cases to (re)generate; default all
    if only:
        return main_selected(tr, vt, mg, only)
    main_selected(tr, vt, mg, None)
    tiny = dict(num_frames=4, img_size=32, patch_size=16, embed_dims=32, num_heads=4,
                num_transformer_layers=2)
    timesformer_case(vt, 'timesformer_tiny', tiny, B=2, seed=0)
    hd64 = dict(num_frames=4, img_size=48, patch_size=16, embed_dims=128, num_heads=2,
                num_transformer_layers=1)
    timesformer_case(vt, 'timesformer_hd64', hd64, B=2, seed=1)
    vv = dict(num_frames_in=8, img_size=32, patch_size=16, embed_dims=32, num_heads=4,
              num_transformer_layers=2)
    vivit_case(vt, 'vivit_tiny_b1', vv, B=1, seed=2)
    vivit_case(vt, 'vivit_tiny_b3', vv, B=3, seed=3)
    space_only_case(vt, 'timesformer_space_only_tiny', tiny, B=2, seed=5)
    space_only_case(vt, 'timesformer_joint_tiny', tiny, B=2, seed=6, attention_type='joint_space_time')
    # 1 + 36*8 = 289 tokens per clip: past the 256-token limit of the single-pass attention kernels (head dim 64)
    joint289 = dict(num_frames=8, img_size=96, patch_size=16, embed_dims=128, num_heads=2, num_transformer_layers=1)
    space_only_case(vt, 'timesformer_joint_n289', joint289, B=1, seed=7, attention_type='joint_space_time')
    mask_cases(mg)
    two_stage = dict(pool_q_stride_size=((1, 1, 2, 2), (3, 1, 2, 2)), feature_dim=216)     # model_trainer.py:54
    maskfeat_case(vt, 'maskfeat_s32', dict(img_size=32, num_frames=8, **two_stage), B=2, seed=7)
    maskfeat_case(vt, 'maskfeat_s64', dict(img_size=64, num_frames=4, **two_stage), B=1, seed=8)
    # MaskFeat.__init__ defaults (three Q-pool stages, video_transformer.py:821): configuration logic only
    maskfeat_case(vt, 'maskfeat_s64_3stage',
                  dict(img_size=64, num_frames=4, feature_dim=2 * 108,
                       pool_q_stride_size=((1, 1, 2, 2), (3, 1, 2, 2), (14, 1, 2, 2))), B=1, seed=9, with_grads=False)


def mixup_cases():
    """Reference Mixup (mixup.py:58-126) under np.random.seed: per seed the mixed float clip, the soft targets and the
    draw (lam / cutmix box recovered by replaying the reference's own helper calls on a copy of the RNG state)."""
    sys.path.insert(0, REF)
    import mixup as ref_mixup
    rows = {}
    B, T, C, H, W, NC = 4, 2, 3, 32, 32, 7
    seeds = list(range(12))
    for seed in seeds:
        g = torch.Generator().manual_seed(seed)
        u8 = torch.randint(0, 256, (B, T, H, W, C), generator=g, dtype=torch.uint8)
        labels = torch.randint(0, NC, (B,), generator=g)
        x = ((u8.float() / 255.0 - 0.45) / 0.225).permute(0, 1, 4, 2, 3).contiguous()      # ToTensor + Normalize
        np.random.seed(seed)
        fn = ref_mixup.Mixup(num_classes=NC)
        xm, tgt = fn(x.clone(), labels)
        rows[f'u8_{seed}'] = u8.numpy()
        rows[f'labels_{seed}'] = labels.numpy()
        rows[f'mixed_{seed}'] = xm.numpy()
        rows[f'target_{seed}'] = tgt.cpu().numpy()
    # reference one_hot defaults to device='cuda'; Mixup passes x.device, so CPU works
    rows['seeds'] = np.asarray(seeds)
    rows['num_classes'] = np.int64(NC)
    np.savez_compressed(os.path.join(GOLD, 'mixup.npz'), **rows)
    print(f'[mixup] {len(seeds)} seeds stored from the reference Mixup class')


def checkpoint_remap_cases():
    """The reference's pretrain_pth loaders (weight_init.py:107-314) on the synthetic checkpoints of
    tests/test_checkpoint_loaders.py: per case the key set of the state dict handed to load_state_dict and, per key, the
    shape and a SHA-256 prefix of the tensor bytes (the remaps are copies / repeats / scalings, compared bit for bit)."""
    import json
    from tests import test_checkpoint_loaders as T
    sys.path.insert(0, REF)
    import weight_init as ref_wi

    class Catch(torch.nn.Module):
        """stands in for the model: records the state dict the reference loader hands to load_state_dict"""
        def load_state_dict(self, sd, strict=True):
            self.got = dict(sd)
            return torch.nn.modules.module._IncompatibleKeys([], [])

    rows = {}
    with tempfile.TemporaryDirectory() as d:
        for conv_type, attention_type, copy_strategy, extend in T.REMAP_CASES:
            for kind, make, ref_fn, inner in (('vit', T._vit_image_checkpoint, ref_wi.init_from_vit_pretrain_, 'state_dict'),
                                              ('mae', T._mae_checkpoint, ref_wi.init_from_mae_pretrain_, 'model')):
                path = os.path.join(d, f'{kind}.pth')
                torch.save({inner: make()}, path)
                catch = Catch()
                ref_fn(catch, path, conv_type, attention_type, copy_strategy, extend, 2, 1)
                rows[T.remap_case_id(kind, conv_type, attention_type, copy_strategy, extend)] = T.state_digest(catch.got)
    sd = T._kinetics_checkpoint()
    ref_wi.replace_state_dict(sd)
    rows['kinetics'] = T.state_digest(sd)
    with open(os.path.join(GOLD, 'checkpoint_remaps.json'), 'w') as fh:          # one line per case
        fh.write('{\n' + ',\n'.join(f'{json.dumps(c)}: {json.dumps(rows[c], sort_keys=True)}' for c in sorted(rows)) + '\n}\n')
    print(f'[checkpoint_remaps] {len(rows)} state dicts from the reference loaders')


def trainer_case():
    """What the reference's model_trainer.py asks of the modules videotransformer_pytorch_b200/shim stands in for: the
    names the reference files import from them, the constructor calls VideoTransformer.__init__ (model_trainer.py:40-104)
    makes for one supervised TimeSformer configuration, and the parameter names / shapes and no-weight-decay keywords of
    the trainer built from the reference's own modules."""
    import ast
    import importlib
    import json
    from tests.test_shim import SHIM, SHIM_MODULES, TRAINER_CFG

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m

    class Accuracy:
        def __init__(self, *a, **k):
            pass

    stub('pytorch_lightning', LightningModule=torch.nn.Module)
    stub('pytorch_lightning.utilities')
    stub('pytorch_lightning.utilities.distributed', rank_zero_only=lambda f: f)
    stub('torchmetrics', Accuracy=Accuracy)
    stub('timm'); stub('timm.loss', SoftTargetCrossEntropy=torch.nn.CrossEntropyLoss)
    stub('matplotlib'); stub('matplotlib.pyplot')
    from oracle.pytorchvideo_restated import install_stub_modules
    install_stub_modules()
    imports = {}
    for f in sorted(os.listdir(REF)):
        if f.endswith('.py'):
            with open(os.path.join(REF, f)) as fh:
                for node in ast.walk(ast.parse(fh.read())):
                    if isinstance(node, ast.ImportFrom) and node.level == 0 and node.module in SHIM_MODULES:
                        imports.setdefault(node.module, set()).update(a.name for a in node.names)
    cfg = types.SimpleNamespace(**TRAINER_CFG)
    saved_path = list(sys.path)

    def fresh_trainer(first):
        for k in SHIM_MODULES + ('model_trainer', 'utils', 'optimizer', 'weight_init'):
            sys.modules.pop(k, None)
        sys.path[:] = first + [REF] + saved_path
        return importlib.import_module('model_trainer')

    # with the shim first on sys.path: record every model / head constructor call the trainer makes
    calls = []
    fresh_trainer([SHIM])
    for mod, name in (('video_transformer', 'TimeSformer'), ('video_transformer', 'ViViT'), ('video_transformer', 'MaskFeat'),
                      ('transformer', 'ClassificationHead')):
        cls = getattr(sys.modules[mod], name)
        setattr(sys.modules[mod], name, lambda *a, _n=name, _c=cls, **k: calls.append([_n, list(a), k]) or _c(*a, **k))
    sys.modules.pop('model_trainer')
    importlib.import_module('model_trainer').VideoTransformer(cfg, trainer=None, ckpt_dir='.', do_eval=False, do_test=False)
    # the reference's own modules: the parameter surface the trainer (and its optimizer grouping) sees
    torch.manual_seed(0)
    vt_ref = fresh_trainer([]).VideoTransformer(cfg, trainer=None, ckpt_dir='.', do_eval=False, do_test=False)
    sys.path[:] = saved_path
    row = {'cfg': TRAINER_CFG, 'imports': {k: sorted(v) for k, v in sorted(imports.items())}, 'constructions': calls,
           'named_parameters': [[n, list(p.shape)] for n, p in vt_ref.named_parameters()],
           'no_weight_decay_keywords': sorted(vt_ref.no_weight_decay_keywords())}
    with open(os.path.join(GOLD, 'reference_trainer.json'), 'w') as fh:          # one line per entry / parameter
        fh.write('{\n' + ',\n'.join(f'{json.dumps(k)}: ' + ('[\n' + ',\n'.join(json.dumps(e) for e in v) + '\n]'
                                                            if k == 'named_parameters' else json.dumps(v))
                                     for k, v in row.items()) + '\n}\n')
    print(f'[reference_trainer] {len(calls)} constructor calls, {len(row["named_parameters"])} parameters')


def main_selected(tr, vt, mg, only):
    """Cases added after round 1 (run alone with `python oracle/make_golden.py <name> ...`)."""
    want = lambda n: only is None or n in only
    vv = dict(num_frames_in=8, img_size=32, patch_size=16, embed_dims=32, num_heads=4, num_transformer_layers=2)
    if want('vivit_joint_tiny'):
        vivit_variant_case(vt, 'vivit_joint_tiny', vv, B=2, seed=11, attention_type='joint_space_time')
    if want('vivit_divided_tiny'):
        vivit_variant_case(vt, 'vivit_divided_tiny', vv, B=2, seed=12, attention_type='divided_space_time')
    vv128 = dict(num_frames_in=8, img_size=48, patch_size=16, embed_dims=128, num_heads=2, num_transformer_layers=1)
    if want('vivit_joint_hd64'):        # D = 128: the width the GPU row-map LayerNorm needs (D % 128 == 0)
        vivit_variant_case(vt, 'vivit_joint_hd64', vv128, B=2, seed=13, attention_type='joint_space_time')
    if want('vivit_divided_hd64'):
        vivit_variant_case(vt, 'vivit_divided_hd64', vv128, B=2, seed=14, attention_type='divided_space_time')
    if want('mixup'):
        mixup_cases()
    if want('checkpoint_remaps'):
        checkpoint_remap_cases()
    if want('reference_trainer'):
        trainer_case()


if __name__ == '__main__':
    main()
