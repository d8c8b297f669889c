"""TimeSformer at input sizes other than img_size on the B200: the bicubic position-table kernels against F.interpolate,
the models against the reference goldens, divided spatial attention past 256 tokens per frame (448^2 frames: 785 tokens),
and a captured training step at 448^2.  -m gpu"""
import math

import pytest
import torch
import torch.nn.functional as F

from tests.conftest import check_grads, rel_err

pytestmark = pytest.mark.gpu

# reference-under-bf16-autocast error vs fp64 of TimeSformer-B built at 224 and fed one 8x448^2 clip (train mode + CE),
# measured with `python tools/ref_autocast_error.py timesformer 1 448` (CPU): feature 9.40e-3, loss 3.59e-4, worst parameter
# gradient 1.42e-2, median 8.56e-3
REF_AUTOCAST_448 = dict(feature=9.40e-3, grad_worst=1.42e-2)


def _table_and_scales(side, rows, cols, D, seed):
    g = torch.Generator().manual_seed(seed)
    table = torch.randn(1 + side * side, D, generator=g)
    sf_r, sf_c = (rows + 0.1) / side, (cols + 0.1) / side       # scale factors as interpolate_pos_encoding forms them
    assert (math.floor(side * sf_r), math.floor(side * sf_c)) == (rows, cols)
    return table, sf_r, sf_c


def _reference(table, side, sf_r, sf_c):
    """fp64 F.interpolate of the patch rows (cls row passes through)."""
    D = table.shape[1]
    grid = table[1:].reshape(1, side, side, D).permute(0, 3, 1, 2)
    out = F.interpolate(grid, scale_factor=(sf_r, sf_c), mode='bicubic')
    return torch.cat((table[:1], out.permute(0, 2, 3, 1).reshape(-1, D)))


@pytest.mark.parametrize('side,rows,cols', [(14, 28, 28), (14, 16, 16), (14, 7, 7), (14, 28, 14), (4, 6, 6)])
def test_pos_interp_kernels_vs_f_interpolate_fp64(side, rows, cols):
    from videotransformer_pytorch_b200 import _lib
    k = _lib.K
    table, sf_r, sf_c = _table_and_scales(side, rows, cols, 768, seed=side * 100 + rows)
    got = k.pos_interp_fwd(table.cuda(), side, rows, cols, 1.0 / sf_r, 1.0 / sf_c)
    ref = _reference(table.double(), side, sf_r, sf_c)
    e_f = rel_err(got.cpu(), ref)
    assert torch.equal(got[0].cpu(), table[0])
    # adjoint against fp64 autograd through the same F.interpolate
    dout = torch.randn(1 + rows * cols, 768, generator=torch.Generator().manual_seed(7))
    t64 = table.double().requires_grad_(True)
    (_reference(t64, side, sf_r, sf_c) * dout.double()).sum().backward()
    d1 = k.pos_interp_bwd(dout.cuda(), side, rows, cols, 1.0 / sf_r, 1.0 / sf_c)
    d2 = k.pos_interp_bwd(dout.cuda(), side, rows, cols, 1.0 / sf_r, 1.0 / sf_c)
    torch.cuda.synchronize()
    e_b = rel_err(d1.cpu(), t64.grad)
    print(f'pos interp {side}->{rows}x{cols}: forward rel-L2 {e_f:.2e}, adjoint {e_b:.2e}')
    assert e_f <= 1e-6 and e_b <= 1e-6
    assert torch.equal(d1, d2)                                    # gather form: deterministic


CASES = ['timesformer_interp_down', 'timesformer_interp_joint', 'timesformer_interp_nonsquare',
         'timesformer_interp_space_only', 'timesformer_interp_up']


@pytest.mark.parametrize('name', CASES)
def test_timesformer_interp_golden_eval_and_train(name):
    """The tolerances of test_gpu_modules.py::test_timesformer_hd64_golden_eval_and_train; pos_embed's gradient included."""
    from oracle import interp_oracle as IO
    from tests.conftest import GOLD
    from videotransformer_pytorch_b200 import TimeSformer
    g = IO.load_golden(name, GOLD)
    c = g.cfg
    m = TimeSformer(num_frames=c['num_frames'], img_size=c['img_size'], patch_size=c['patch_size'],
                    embed_dims=c['embed_dims'], num_heads=c['num_heads'],
                    num_transformer_layers=c['num_transformer_layers'], attention_type=g.attention_type)
    m.load_state_dict(g.sd, strict=True)
    m = m.cuda().eval()
    x = g.x.cuda()
    with torch.no_grad():
        y = m(x)
        tok, _ = m.prepare_tokens(x)
        attn = m.get_last_selfattention(x)
    e_tok, e_y, e_attn = rel_err(tok.cpu(), g.out['tokens']), rel_err(y.cpu(), g.out['y_eval']), rel_err(attn.cpu(), g.out['last_attn'])
    print(f'{name}: tokens {e_tok:.2e}  y_eval {e_y:.2e}  last_attn {e_attn:.2e}')
    assert e_tok < 3e-3 and e_y < 1.5e-2 and e_attn < 1e-2
    m.train()
    xg = x.clone().requires_grad_(True)
    torch.manual_seed(g.train_seed)
    yt = m(xg)
    e_tr = rel_err(yt.detach().cpu(), g.out['y_train'])
    (yt.double() * g.out['loss_w'].cuda()).sum().backward()
    e_dx = rel_err(xg.grad.cpu(), g.out['dx'])
    print(f'{name}: y_train {e_tr:.2e}  dx {e_dx:.2e}  pos_embed grad {rel_err(m.pos_embed.grad.cpu(), g.grad["pos_embed"]):.2e}')
    assert e_tr < 1.5e-2 and e_dx < 3e-2
    assert 'pos_embed' in g.grad
    check_grads({n: p.grad for n, p in m.named_parameters()}, g, 3e-2)


def test_spatial_block_at_hr_shape_vs_fp64_oracle():
    """TimeSformer-HR spatial pass: D 768, H 12, T 16, P 784 (785 tokens per frame, streaming kernels), forward and
    backward vs the fp64 oracle; DESIGN §3's per-block contract on the output."""
    from oracle import vt_oracle as O
    from videotransformer_pytorch_b200 import DividedSpatialAttentionWithPreNorm
    torch.manual_seed(0)
    B, T, P, D, H = 1, 16, 784, 768, 12
    blk = DividedSpatialAttentionWithPreNorm(D, H, T, use_cls_token=True, layer_drop=dict(type=None, dropout_p=0.))
    with torch.no_grad():
        for p in blk.parameters():
            p.add_(torch.randn_like(p) * 0.02)
    x = torch.randn(B, 1 + P * T, D)
    w = torch.randn(B, 1 + P * T, D)
    blk = blk.cuda()
    xg = x.cuda().requires_grad_(True)
    y = blk(xg)
    (y * w.cuda()).sum().backward()
    torch.cuda.synchronize()
    sd = {'n.' + k: v.detach().cpu().double().requires_grad_(True) for k, v in blk.state_dict().items()}
    xo = x.double().requires_grad_(True)
    yo = O.divided_spatial(xo, sd, 'n.', T, H, 0.0, False)
    (yo * w.double()).sum().backward()
    e_y, e_dx = rel_err(y.detach().cpu(), yo.detach()), rel_err(xg.grad.cpu(), xo.grad)
    e_g = {k: rel_err(v.grad.cpu(), sd['n.' + k].grad) for k, v in blk.named_parameters()}
    print(f'spatial block 16x785 tokens: output rel-L2 {e_y:.2e}, dx {e_dx:.2e}, worst parameter gradient '
          f'{max(e_g.values()):.2e} ({max(e_g, key=e_g.get)})')
    assert e_y <= 1e-3
    assert e_dx < 1e-2 and max(e_g.values()) < 1e-2


def test_timesformer_b_224_model_on_448_clip_train_step_vs_oracle():
    """TimeSformer-B built at 224, fed one 8x448^2 clip (pos_embed 14x14 -> 28x28, 785-token spatial pass) in train mode
    with cross-entropy, vs the fp32 CPU oracle; gates at 1.5x the reference's own bf16-autocast error at this shape."""
    from oracle import interp_oracle as IO
    from oracle import vt_oracle as O
    from tests.test_gpu_baseline_shapes import NUM_CLASSES, _grad_report, _head, _threads
    from videotransformer_pytorch_b200 import ClassificationHead, TimeSformer
    _threads()
    cfg = dict(O.TIMESFORMER_B)
    sd = O.random_timesformer_state(cfg, seed=0)
    hw, hb = _head()
    g = torch.Generator().manual_seed(2)
    x = torch.randn(1, 8, 3, 448, 448, generator=g)
    y = torch.randint(0, NUM_CLASSES, (1,), generator=g)
    m = TimeSformer(num_frames=8, img_size=224, patch_size=16, embed_dims=768, num_heads=12, num_transformer_layers=12)
    m.load_state_dict(sd, strict=True)
    head = ClassificationHead(NUM_CLASSES, 768)
    head.load_state_dict({'cls_head.weight': hw, 'cls_head.bias': hb}, strict=True)
    m, head = m.cuda().train(), head.cuda().train()
    torch.manual_seed(7)
    feat = m(x.cuda())
    F.cross_entropy(head(feat), y.cuda()).backward()
    torch.cuda.synchronize()

    s = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    hwr, hbr = hw.clone().requires_grad_(True), hb.clone().requires_grad_(True)
    torch.manual_seed(7)
    feat_o = IO.forward(s, x, cfg, 'divided_space_time', training=True)
    F.cross_entropy(feat_o @ hwr.t() + hbr, y).backward()
    e_f = rel_err(feat.detach().cpu(), feat_o.detach())
    named = {n: p.grad for n, p in m.named_parameters()}
    named['cls_head.weight'], named['cls_head.bias'] = head.cls_head.weight.grad, head.cls_head.bias.grad
    ref = {k: v.grad for k, v in s.items()}
    ref['cls_head.weight'], ref['cls_head.bias'] = hwr.grad, hbr.grad
    worst, median, _ = _grad_report('TimeSformer-B 224 model, 8x448 clip', named, ref)
    ac = REF_AUTOCAST_448
    print(f'TimeSformer-B 224 model on 8x448^2: feature rel-L2 {e_f:.2e} (reference under bf16 autocast {ac["feature"]:.2e}), '
          f'pos_embed grad {rel_err(named["pos_embed"].cpu(), ref["pos_embed"]):.2e}')
    assert e_f < 1.5 * ac['feature']
    assert worst < 1.5 * ac['grad_worst']


def test_graphed_step_at_448_matches_eager():
    """The interpolation and the streaming spatial attention inside a captured training step (model built at 224)."""
    from videotransformer_pytorch_b200 import ClassificationHead, TimeSformer
    from videotransformer_pytorch_b200.graph import GraphedTrainStep

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.model = TimeSformer(num_frames=2, img_size=224, patch_size=16, embed_dims=128, num_heads=2,
                                     num_transformer_layers=2)
            self.head = ClassificationHead(10, 128)
            with torch.no_grad():
                for n, p in self.model.named_parameters():
                    if 'temporal_fc' in n:
                        p.normal_(std=0.05)

        def forward(self, x, y):
            return F.cross_entropy(self.head(self.model(x)), y)

    torch.manual_seed(0)
    net = Net().cuda().train()
    x = torch.randn(2, 2, 3, 448, 448).cuda()
    y = torch.tensor([1, 7]).cuda()
    step = GraphedTrainStep(net, (x, y))
    x2 = torch.randn(2, 2, 3, 448, 448).cuda()
    torch.manual_seed(123)
    loss_g = float(step(x2, y).detach())
    gg = {n: p.grad.clone() for n, p in net.named_parameters()}
    for p in net.parameters():
        p.grad = None
    torch.manual_seed(123)
    loss_e = net(x2, y)
    loss_e.backward()
    assert abs(loss_g - float(loss_e)) < 1e-5, (loss_g, float(loss_e))
    bad = [n for n, p in net.named_parameters() if not torch.allclose(gg[n], p.grad, rtol=1e-4, atol=1e-6)]
    assert not bad, (len(bad), bad[:10])
    assert net.model.pos_embed.grad.abs().sum() > 0


def test_vivit_divided_at_img_256_vs_oracle():
    """ViViT model 3 built at 256 (1 + 256 = 257 tokens per spatial pass, streaming kernels), forward and backward."""
    from oracle import vt_oracle as O
    from videotransformer_pytorch_b200 import ViViT
    torch.manual_seed(0)
    cfg = dict(num_frames_in=4, img_size=256, patch_size=16, embed_dims=128, num_heads=2, num_transformer_layers=1)
    m = ViViT(num_frames=4, img_size=256, patch_size=16, embed_dims=128, num_heads=2, num_transformer_layers=1,
              attention_type='divided_space_time')
    with torch.no_grad():
        for n, p in m.named_parameters():
            if 'norm' in n or n.endswith('bias') or 'temporal_fc' in n:
                p.add_(torch.randn_like(p) * 0.05)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    x = torch.randn(2, 4, 3, 256, 256)
    m = m.cuda().eval()
    with torch.no_grad():
        e_eval = rel_err(m(x.cuda()).cpu(), O.vivit_variant_forward({k: v.double() for k, v in sd.items()}, x.double(), cfg,
                                                                     'divided_space_time'))
    m.train()
    torch.manual_seed(3)
    yt = m(x.cuda())
    w = torch.randn(yt.shape)
    (yt * w.cuda()).sum().backward()
    s = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    torch.manual_seed(3)
    yo = O.vivit_variant_forward(s, x.double(), cfg, 'divided_space_time', training=True)
    (yo * w.double()).sum().backward()
    e_tr = rel_err(yt.detach().cpu(), yo.detach())
    errs = {n: rel_err(p.grad.cpu(), s[n].grad) for n, p in m.named_parameters()}
    print(f'ViViT divided 256^2: eval {e_eval:.2e}, train {e_tr:.2e}, worst grad {max(errs.values()):.2e} '
          f'({max(errs, key=errs.get)})')
    assert e_eval < 1.5e-2 and e_tr < 1.5e-2 and max(errs.values()) < 3e-2
