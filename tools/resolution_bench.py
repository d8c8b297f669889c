"""Training-step time of TimeSformer-B (+ classification head + cross-entropy) at three input resolutions on one GPU.

    python tools/resolution_bench.py [--batch 8] [--batch-448 4] [--batch-hr 2] [--steps 10] [--warmup 3] [--min-seconds 1]

Configurations (per-GPU batch per flag):
  224      model built at 224, 8 x 224^2 clips              (the bench.py headline workload)
  448      model built at 224, 8 x 448^2 clips              (pos_embed resampled 14x14 -> 28x28; 785 tokens per frame)
  hr       TimeSformer-HR: model built at 448, 16 x 448^2   (785 tokens per frame, 16 frames)
Each line times the CUDA-graph captured fwd+bwd step with CUDA events over a window of at least --min-seconds after
warm-up, and reports the algorithmic FLOP per clip (from the shapes, below), the whole step's share of the measured bf16
peak in MEASURED_PEAKS.json ("not measured" when that file is absent), the card and its power limit.  A second capture of
the same step with CUDA-event nodes around every spatial-attention launch gives their in-situ time per step.
Writes nothing; needs a CUDA device.
"""
import argparse
import json
import math
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

NUM_CLASSES, D, HEADS, LAYERS, PATCH = 400, 768, 12, 12, 16
CONFIGS = {'224': dict(img_size=224, frames=8, size=224), '448': dict(img_size=224, frames=8, size=448),
           'hr': dict(img_size=448, frames=16, size=448)}


def flop_per_clip(T, size):
    """Algorithmic FLOP of one clip's forward through TimeSformer-B divided space-time attention (2 per multiply-add;
    attention cores 4 N^2 d per sequence), times 3 for forward + backward.  At 8 x 224^2: 391.66 GFLOP forward."""
    P = (size // PATCH) ** 2
    S = 1 + P * T
    patch = 2 * T * P * D * 3 * PATCH * PATCH
    temporal = 2 * P * T * D * 3 * D + 4 * P * T * T * D + 2 * 2 * P * T * D * D
    spatial = 2 * T * (P + 1) * D * 3 * D + 4 * T * (P + 1) ** 2 * D + 2 * T * (P + 1) * D * D
    ffn = 2 * 2 * S * D * 4 * D
    head = 2 * D * NUM_CLASSES
    return 3 * (patch + LAYERS * (temporal + spatial + ffn) + head), P


def peak_tflops():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as fh:
            return float(json.load(fh)['bf16_tflops_sustained'])
    except Exception:
        return None


def card():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i',
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        power = out or 'not measured'
    except Exception:
        power = 'not measured'
    return name, power


class Step(torch.nn.Module):
    def __init__(self, img_size, frames):
        super().__init__()
        from videotransformer_pytorch_b200 import ClassificationHead, TimeSformer
        self.model = TimeSformer(num_frames=frames, img_size=img_size, patch_size=PATCH, embed_dims=D, num_heads=HEADS,
                                 num_transformer_layers=LAYERS, attention_type='divided_space_time')
        self.cls_head = ClassificationHead(NUM_CLASSES, D, eval_metrics='finetune')
        with torch.no_grad():   # temporal_fc is zero-init in the reference: make the branch live (as bench.py does)
            for n, p in self.model.named_parameters():
                if 'temporal_fc' in n:
                    p.normal_(std=0.02)

    def forward(self, x, y):
        return self.cls_head.loss(self.model(x), y)


def spatial_attention_ms(net, inputs, P):
    """In-situ time per step of the spatial-attention launches (sequence length P + 1), bench.py's gemm_probe technique:
    the step captured once more with external CUDA-event nodes around each such launch, then replayed."""
    from videotransformer_pytorch_b200 import _lib
    from videotransformer_pytorch_b200.graph import GraphedTrainStep
    K = _lib.K
    orig = {n: getattr(K, n) for n in ('attn_fwd', 'attn_bwd', 'xattn_fwd', 'xattn_bwd')}
    rec = []

    def bracket(fn, *a, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True)
        e0.record()
        out = fn(*a, **kw)
        e1.record()
        rec.append((e0, e1))
        return out

    def attn_fwd(qkv, Bp, N, *a, **kw):
        f = orig['attn_fwd']
        return bracket(f, qkv, Bp, N, *a, **kw) if N == P + 1 else f(qkv, Bp, N, *a, **kw)

    def attn_bwd(qkv, ctx, dctx, lse, Bp, N, *a, **kw):
        f = orig['attn_bwd']
        return bracket(f, qkv, ctx, dctx, lse, Bp, N, *a, **kw) if N == P + 1 else f(qkv, ctx, dctx, lse, Bp, N, *a, **kw)

    def xattn_fwd(q, *a, **kw):
        f = orig['xattn_fwd']
        return bracket(f, q, *a, **kw) if q.shape[2] == P + 1 else f(q, *a, **kw)

    def xattn_bwd(q, *a, **kw):
        f = orig['xattn_bwd']
        return bracket(f, q, *a, **kw) if q.shape[2] == P + 1 else f(q, *a, **kw)

    K.attn_fwd, K.attn_bwd, K.xattn_fwd, K.xattn_bwd = attn_fwd, attn_bwd, xattn_fwd, xattn_bwd
    try:
        probe = GraphedTrainStep(net, inputs, warmup=0)      # captures the bracketed launches once
        for _ in range(2):
            probe(*inputs)
        torch.cuda.synchronize()
    finally:
        for n, f in orig.items():
            setattr(K, n, f)
    return sum(a.elapsed_time(b) for a, b in rec), len(rec)


def run(name, B, args, name_power):
    from videotransformer_pytorch_b200.graph import GraphedTrainStep
    cfg = CONFIGS[name]
    T, size = cfg['frames'], cfg['size']
    flop, P = flop_per_clip(T, size)
    line = dict(config=name, model_img_size=cfg['img_size'], clip=f'{B}x{T}x3x{size}x{size}', batch=B, tokens_per_frame=P + 1,
                flop_per_clip=flop, gpu=name_power[0], power_limit=name_power[1])
    try:
        torch.manual_seed(0)
        net = Step(cfg['img_size'], T).cuda().train()
        g = torch.Generator().manual_seed(100)
        inputs = (torch.randn(B, T, 3, size, size, generator=g).cuda(), torch.randint(0, NUM_CLASSES, (B,), generator=g).cuda())
        step = GraphedTrainStep(net, inputs, warmup=3)
        for _ in range(args.warmup):
            step(*inputs)
        torch.cuda.synchronize()

        def window(k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(k):
                step(*inputs)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)
        k = args.steps
        ms = window(k)
        if ms < args.min_seconds * 1e3:                    # stretch the window to at least min_seconds
            k = max(k, math.ceil(k * args.min_seconds * 1e3 / ms * 1.1))
            ms = window(k)
        ms_step = ms / k
        pk = peak_tflops()
        achieved = flop * B / (ms_step * 1e-3) / 1e12
        line.update(ms_per_step=ms_step, clips_per_s=B / (ms_step * 1e-3), steps_timed=k, window_s=ms / 1e3,
                    achieved_tflops=achieved,
                    whole_step_frac_of_bf16_peak=(achieved / pk) if pk else 'not measured (no MEASURED_PEAKS.json)',
                    bf16_peak_tflops=pk if pk else 'not measured')
        del step
        sp_ms, n = spatial_attention_ms(net, inputs, P)
        line.update(spatial_attention_ms_per_step=sp_ms, spatial_attention_launches=n,
                    spatial_attention_frac_of_step=sp_ms / ms_step,
                    spatial_attention_kernels='vt_attn_fwd/bwd (single pass)' if P + 1 <= 256 else
                    'vt_xattn_fwd/bwd (streaming; the fp32 dk/dv copy-back after xattn_bwd is not included)')
    except torch.cuda.OutOfMemoryError as exc:
        line.update(ms_per_step='not measured', error=f'out of memory at batch {B}: {str(exc)[:160]}')
    finally:
        torch.cuda.empty_cache()
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--batch', type=int, default=8, help='clips per GPU at 8 x 224^2')
    ap.add_argument('--batch-448', type=int, default=4, help='clips per GPU at 8 x 448^2 (model built at 224)')
    ap.add_argument('--batch-hr', type=int, default=2, help='clips per GPU for TimeSformer-HR 16 x 448^2')
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--min-seconds', type=float, default=1.0)
    ap.add_argument('--configs', default='224,448,hr')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('resolution_bench.py: no CUDA device; step times are only measured on the GPU')
    from videotransformer_pytorch_b200 import _lib
    _lib.load_library()
    name_power = card()
    batches = {'224': args.batch, '448': args.batch_448, 'hr': args.batch_hr}
    for name in args.configs.split(','):
        run(name, batches[name], args, name_power)


if __name__ == '__main__':
    main()
