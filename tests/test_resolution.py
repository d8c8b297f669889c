"""TimeSformer at input sizes other than img_size (bicubic pos_embed interpolation, reference video_transformer.py:171-191)
and divided spatial attention past 256 tokens per frame, on the CPU: the oracle against goldens recorded from the reference,
the package's host logic on the emulated kernel table, the params struct of the new kernels, and the rejected sizes."""
import math

import pytest
import torch

from tests.conftest import GOLD, check_grads, rel_err
from tests.emu_kernels import EmuKernels

CASES = ['timesformer_interp_down', 'timesformer_interp_joint', 'timesformer_interp_nonsquare',
         'timesformer_interp_space_only', 'timesformer_interp_up']


class PosInterpEmu(EmuKernels):
    """The CPU kernel emulation plus vt_pos_interp_fwd/bwd: dense 1-D weight matrices built from the scalar parameters
    exactly as the kernels build them (fp32 scales, 4 clamped cubic taps with A = -0.75, repeated border taps added)."""

    @staticmethod
    def _cubic_matrix(n_out, n_in, scale):
        A = -0.75
        sc = float(torch.tensor(scale, dtype=torch.float32))
        conv1 = lambda x: ((A + 2) * x - (A + 3)) * x * x + 1
        conv2 = lambda x: ((A * x - 5 * A) * x + 8 * A) * x - 4 * A
        W = torch.zeros(n_out, n_in, dtype=torch.float64)
        for i in range(n_out):
            src = (i + 0.5) * sc - 0.5
            i0 = math.floor(src)
            t = src - i0
            for k, wk in enumerate((conv2(t + 1), conv1(t), conv1(1 - t), conv2(2 - t))):
                W[i, min(max(i0 - 1 + k, 0), n_in - 1)] += wk
        return W

    def pos_interp_fwd(self, table, side, rows, cols, scale_r, scale_c):
        self.calls.append(('pos_interp_fwd', side, rows, cols))
        t = self._up(table)
        D = t.shape[1]
        Wr = self._cubic_matrix(rows, side, scale_r).to(t.dtype)
        Wc = self._cubic_matrix(cols, side, scale_c).to(t.dtype)
        g = torch.einsum('ia,abd,jb->ijd', Wr, t[1:].reshape(side, side, D), Wc)
        return torch.cat((t[:1], g.reshape(rows * cols, D))).to(self.f)

    def pos_interp_bwd(self, dout, side, rows, cols, scale_r, scale_c):
        d = self._up(dout)
        D = d.shape[1]
        Wr = self._cubic_matrix(rows, side, scale_r).to(d.dtype)
        Wc = self._cubic_matrix(cols, side, scale_c).to(d.dtype)
        g = torch.einsum('ia,ijd,jb->abd', Wr, d[1:].reshape(rows, cols, D), Wc)
        return torch.cat((d[:1], g.reshape(side * side, D))).to(self.f)


@pytest.fixture
def emu():
    """Swap the kernel table for the CPU emulation with the position-table kernels."""
    from videotransformer_pytorch_b200 import _lib
    old = _lib.K
    _lib.K = PosInterpEmu(exact=True)
    yield _lib.K
    _lib.K = old


_CACHE = {}


def golden(name):
    from oracle import interp_oracle as IO
    if name not in _CACHE:
        _CACHE[name] = IO.load_golden(name, GOLD)
    return _CACHE[name]


def build(g, **kw):
    from videotransformer_pytorch_b200 import TimeSformer
    c = g.cfg
    m = TimeSformer(num_frames=c['num_frames'], img_size=c['img_size'], patch_size=c['patch_size'],
                    embed_dims=c['embed_dims'], num_heads=c['num_heads'],
                    num_transformer_layers=c['num_transformer_layers'], attention_type=g.attention_type, **kw)
    m.load_state_dict(g.sd, strict=True)
    return m


@pytest.mark.parametrize('name', CASES)
def test_oracle_vs_interp_golden(name):
    from oracle import interp_oracle as IO
    g = golden(name)
    at = g.attention_type
    sd = {k: v.double() for k, v in g.sd.items()}
    x = g.x.double()
    with torch.no_grad():
        assert rel_err(IO.forward(sd, x, g.cfg, at), g.out['y_eval']) < 1e-12
        assert rel_err(IO.tokens(sd, x, g.cfg, at), g.out['tokens']) < 1e-12
        assert rel_err(IO.last_selfattention(sd, x, g.cfg, at), g.out['last_attn']) < 1e-12
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xg = x.clone().requires_grad_(True)
    torch.manual_seed(g.train_seed)
    y = IO.forward(sdg, xg, g.cfg, at, training=True)
    assert rel_err(y, g.out['y_train']) < 1e-12
    (y * g.out['loss_w']).sum().backward()
    assert rel_err(xg.grad, g.out['dx']) < 1e-6          # golden dx stored as fp32
    check_grads({k: v.grad for k, v in sdg.items()}, g, 1e-6)


def test_interp_oracle_is_vt_oracle_at_the_model_size():
    """At the model's own size the interpolation is the identity: the same numbers as vt_oracle's TimeSformer."""
    from oracle import interp_oracle as IO
    from oracle import vt_oracle as O
    from tests.conftest import Golden
    g = Golden('timesformer_hd64')
    sd = {k: v.double() for k, v in g.sd.items()}
    x = g.x.double()
    with torch.no_grad():
        assert torch.equal(IO.forward(sd, x, g.cfg, 'divided_space_time'), O.timesformer_forward(sd, x, g.cfg))
        assert torch.equal(IO.tokens(sd, x, g.cfg, 'divided_space_time'), O.timesformer_tokens(sd, x, g.cfg))


def test_interp_goldens_exercise_the_resampling():
    """Each fixture's clip really takes the interpolation branch, and the non-square one the transposed table."""
    for name in CASES:
        g = golden(name)
        H, W = g.x.shape[-2:]
        assert (H, W) != (g.cfg['img_size'],) * 2
    g = golden('timesformer_interp_nonsquare')
    assert g.x.shape[-2] != g.x.shape[-1]


@pytest.mark.parametrize('name', CASES)
def test_package_vs_interp_golden_on_emulated_kernels(emu, name):
    """Same tolerances as test_host_logic_emu.py applies to the TimeSformer goldens."""
    g = golden(name)
    m = build(g).eval()
    with torch.no_grad():
        y = m(g.x)
        tok, _ = m.prepare_tokens(g.x)
        attn = m.get_last_selfattention(g.x)
    assert rel_err(tok, g.out['tokens']) < 1e-5
    assert rel_err(y, g.out['y_eval']) < 2e-5
    assert attn.shape == g.out['last_attn'].shape
    assert rel_err(attn, g.out['last_attn']) < 2e-5
    assert any(c[0] == 'pos_interp_fwd' for c in emu.calls if isinstance(c, tuple))
    m.train()
    x = g.x.clone().requires_grad_(True)
    torch.manual_seed(g.train_seed)
    y = m(x)
    assert rel_err(y, g.out['y_train']) < 2e-5
    (y.double() * g.out['loss_w']).sum().backward()
    assert rel_err(x.grad, g.out['dx']) < 1e-4
    grads = {n: p.grad for n, p in m.named_parameters()}
    assert all(v is not None for v in grads.values())
    check_grads(grads, g, 2e-4)


def test_interpolate_pos_encoding_matches_reference_semantics(emu):
    """The public method: identity (the very same Parameter) at the model's own size, the oracle's F.interpolate
    otherwise (including the transposed table of a non-square clip)."""
    from oracle import interp_oracle as IO
    g = golden('timesformer_interp_nonsquare')
    m = build(g)
    D = g.cfg['embed_dims']
    assert m.interpolate_pos_encoding(torch.zeros(1, 5, D), 32, 32) is m.pos_embed
    for (h, w) in ((64, 64), (32, 64), (64, 32), (48, 80), (16, 16)):
        npatch = (h // 16) * (w // 16)
        got = m.interpolate_pos_encoding(torch.zeros(1, 1 + npatch, D), w, h)
        ref = IO.interpolate_pos_encoding(g.sd['pos_embed'].double(), npatch, w, h, 16)
        assert got.shape == ref.shape == (1, 1 + npatch, D)
        assert rel_err(got, ref) < 1e-6, (h, w)


def test_sine_cosine_table_is_interpolated_without_gradient(emu):
    from videotransformer_pytorch_b200 import TimeSformer
    torch.manual_seed(0)
    m = TimeSformer(num_frames=2, img_size=32, patch_size=16, embed_dims=64, num_heads=1, num_transformer_layers=1,
                    use_learnable_pos_emb=False)
    x = torch.randn(1, 2, 3, 64, 48)
    pos = m.interpolate_pos_encoding(torch.zeros(1, 1 + 12, 64), 48, 64)
    assert pos.shape == (1, 13, 64) and not pos.requires_grad
    m.train()
    m(x).sum().backward()
    assert m.patch_embed.projection.weight.grad is not None


def test_spatial_attention_past_256_tokens_routes_to_streaming_kernels(emu):
    """img 256 / patch 16: 1 + 256 = 257 tokens per frame in the spatial pass — the streaming kernels, against the oracle."""
    from oracle import vt_oracle as O
    from videotransformer_pytorch_b200 import DividedSpatialAttentionWithPreNorm
    torch.manual_seed(0)
    B, T, P, D, H = 1, 2, 256, 64, 1
    blk = DividedSpatialAttentionWithPreNorm(D, H, T, use_cls_token=True, layer_drop=dict(type=None, dropout_p=0.))
    with torch.no_grad():
        for p in blk.parameters():
            p.add_(torch.randn_like(p) * 0.05)
    x = torch.randn(B, 1 + P * T, D, requires_grad=True)
    y = blk(x)
    w = torch.randn_like(y)
    (y * w).sum().backward()
    assert ('xattn', (B * T, H, P + 1, D // H), P + 1) in emu.calls
    sd = {'n.' + k: v.detach().double().requires_grad_(True) for k, v in blk.state_dict().items()}
    xo = x.detach().double().requires_grad_(True)
    yo = O.divided_spatial(xo, sd, 'n.', T, H, 0.0, False)
    (yo * w.double()).sum().backward()
    assert rel_err(y, yo) < 1e-6
    assert rel_err(x.grad, xo.grad) < 1e-6
    for k, v in blk.named_parameters():
        assert rel_err(v.grad, sd['n.' + k].grad) < 1e-6, k


@pytest.mark.parametrize('B,T,P', [(1, 8, 256), (1, 8, 784), (2, 4, 400)])
@pytest.mark.parametrize('kind', ['temporal', 'spatial'])
def test_residual_epilogue_segments_at_high_resolution_periods(B, T, P, kind):
    """The TMA residual epilogue's walk (tests/test_kernel_algorithms_sim.py) at the patch counts of 256^2, 448^2 and
    320^2 frames."""
    from tests.test_kernel_algorithms_sim import test_residual_epilogue_segments_cover_every_row_once as walk
    walk(B, T, P, kind)


def test_unsupported_sizes_raise(emu):
    from videotransformer_pytorch_b200 import TimeSformer, ViViT
    m = TimeSformer(num_frames=2, img_size=32, patch_size=16, embed_dims=64, num_heads=1, num_transformer_layers=1)
    with pytest.raises(NotImplementedError, match=r'W % 16 == 0'):
        m(torch.randn(1, 2, 3, 32, 40))
    with pytest.raises(NotImplementedError, match=r'H % 16 == 0'):
        m(torch.randn(1, 2, 3, 40, 32))
    with pytest.raises(NotImplementedError, match=r'W % 16 == 0'):
        m(torch.randint(0, 256, (1, 2, 32, 40, 3), dtype=torch.uint8))       # channels-last byte clip: same axes
    narrow = TimeSformer(num_frames=2, img_size=24, patch_size=12, embed_dims=64, num_heads=1, num_transformer_layers=1)
    with pytest.raises(NotImplementedError, match='multiple of 8'):
        narrow(torch.randn(1, 2, 3, 24, 24))
    rect = TimeSformer(num_frames=2, img_size=(32, 64), patch_size=16, embed_dims=64, num_heads=1, num_transformer_layers=1)
    with pytest.raises(NotImplementedError, match='square patch grid'):
        rect(torch.randn(1, 2, 3, 64, 64))
    vv = ViViT(num_frames=4, img_size=32, patch_size=16, embed_dims=64, num_heads=1, num_transformer_layers=1)
    with pytest.raises(NotImplementedError, match='ViViT'):
        vv(torch.randn(1, 4, 3, 64, 64))


def test_byte_clip_reads_height_and_width_from_its_own_axes(emu):
    """uint8 [B, T, H, W, C] at a non-square size gives what the float [B, T, C, H, W] clip gives."""
    g = golden('timesformer_interp_nonsquare')
    m = build(g).eval()
    mean, std = (0.45, 0.45, 0.45), (0.225, 0.225, 0.225)
    m.set_input_normalization(mean, std)
    u8 = torch.randint(0, 256, (2, 2, 32, 64, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(0))
    xf = (u8.float() / 255.0 - torch.tensor(mean)) / torch.tensor(std)
    with torch.no_grad():
        assert rel_err(m(u8), m(xf.permute(0, 1, 4, 2, 3).contiguous())) < 1e-5


def test_pos_interp_params_match_the_header(tmp_path):
    """ctypes mirror of vt_pos_interp_params against the C header (the offsetof check of test_abi.py)."""
    import os
    import shutil
    import subprocess
    from tests.conftest import ROOT
    from videotransformer_pytorch_b200 import _lib
    if not shutil.which('gcc'):
        pytest.skip('no gcc')
    cls = _lib.PosInterpParams
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{os.path.join(ROOT, "include", "vt_b200.h")}"',
             'int main(void) {', '  printf("size %zu\\n", sizeof(vt_pos_interp_params));']
    for fname, _ in cls._fields_:
        cf = 'in' if fname == 'inp' else fname
        lines.append(f'  printf("{fname} %zu\\n", offsetof(vt_pos_interp_params, {cf}));')
    lines += ['  return 0;', '}']
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'layout'
    subprocess.check_call(['gcc', str(src), '-o', str(exe)])
    got = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(got['size']) == __import__('ctypes').sizeof(cls)
    for fname, _ in cls._fields_:
        assert int(got[fname]) == getattr(cls, fname).offset, fname
    assert {'vt_pos_interp_fwd', 'vt_pos_interp_bwd'} <= set(_lib.EXPORTS)
