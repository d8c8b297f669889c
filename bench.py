#!/usr/bin/env python
"""Headline benchmark: clips/sec of the video-transformer forward+backward hot path on N B200 GPUs, next to the
reference algorithm's CPU timing.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload timesformer|vivit|mvit|maskfeat] [--batch B]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference [--steps K --warmup W]      # CPU arm (oracle port of the reference)
    python bench.py --dump-outputs DIR ...                       # also write the last timed step's outputs as DIR/*.npy

One JSON line on stdout (rank 0).  Workloads = BASELINE.json configs:
  timesformer (default, configs 1-2)  TimeSformer-B divided_space_time 8x224x224, batch 8 / GPU, + cls head + CE
  vivit       (config 3)              ViViT-B fact_encoder 16x224x224 (tubelet 2), batch 8 / GPU, + cls head + CE
  mvit        (config 4)              MViT-B 16x224x224 pooling attention (MaskFeat.forward_features), batch 8 / GPU
  maskfeat    (config 5)              MaskFeat MViT-B pretrain step, batch 16 / GPU: CubeMaskGenerator masks, HOG targets
                                      from the HOG kernel, decoder + masked MSE
A "step" = one pass of the hot path over one synthetic batch: forward, loss, full backward, and for N > 1 the bucketed
gradient all-reduce.  The optimizer update is outside the metric (BASELINE.json: fwd+bwd).
  value : inputs resident in HBM before the timed region
  e2e   : same step through the public nn.Module API with the batch copied from pinned host memory every step (for
          maskfeat: the uint8 clips; masks drawn on the host, HOG targets computed on the device inside the region) and the
          loss read back to the host
The default line also carries `other_workloads`: the same measurement for the three other configs.
--dump-outputs DIR writes what the caller of the timed step receives after its last timed step: the loss (loss.npy) and
every parameter gradient (grad.<parameter name>.npy, float32; a gradient of more than DUMP_SAMPLE elements as the same
seeded sample of its flattened elements on every run).  Inputs, weights and DropPath draws are seeded, so two builds run
with the same arguments can be compared array for array.  Split-K GEMMs add their partial sums in an order that varies
from run to run, and the bf16 operand casts downstream can turn such last-bit differences into bf16-rounding ones: compare
gradients with a tolerance, not bit for bit.  The benchmark writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: no __pycache__ written into it

UNIT = 'clips/s'
IMG, NUM_CLASSES = 224, 400
# algorithmic FLOPs per clip, fwd+bwd (SURVEY.md §8d; MAC = 2 FLOP, bwd = 2x fwd)
WORKLOADS = {
    'timesformer': dict(metric='clips/sec (BxTx3x224x224) TimeSformer-B fwd+bwd', frames=8, batch=8, flop_per_clip=1.175e12,
                        desc='TimeSformer-B divided_space_time 8x224x224 fwd+bwd (+cls head, CE), train mode, DropPath 0..0.1'),
    'vivit': dict(metric='clips/sec (BxTx3x224x224) ViViT-B fwd+bwd', frames=16, batch=8, flop_per_clip=0.850e12,
                  desc='ViViT-B fact_encoder 16x224x224 tubelet 2 fwd+bwd (+cls head, CE), train mode, DropPath 0..0.1'),
    'mvit': dict(metric='clips/sec (BxTx3x224x224) MViT-B fwd+bwd', frames=16, batch=8, flop_per_clip=0.515e12,
                 desc='MViT-B 16x224x224 pooling attention (MaskFeat.forward_features, reference 2-stage Q-pool config) fwd+bwd'),
    'maskfeat': dict(metric='clips/sec (BxTx3x224x224) MaskFeat MViT-B pretrain fwd+bwd', frames=16, batch=16, flop_per_clip=0.516e12,
                     desc='MaskFeat MViT-B pretrain step 16x224x224: cube masks, HOG targets (HOG kernel), decoder + masked MSE, fwd+bwd'),
}
DUMP_SAMPLE, DUMP_MAX_BYTES = 1 << 16, 64 << 20
# attention-GEMM subset of the TimeSformer step (north_star): qkv + QK^T + PV + out-proj of both passes, fwd+bwd
MASKFEAT_KW = dict(pool_q_stride_size=[[1, 1, 2, 2], [3, 1, 2, 2]], feature_dim=2 * 2 * 2 * 3 * 9)


def peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as fh:
            p = json.load(fh)
        return dict(tflops=float(p['bf16_tflops_sustained']), burst=float(p['bf16_tflops']), hbm=float(p['hbm_gbs']),
                    source='measured (MEASURED_PEAKS.json, sustained bf16)')
    except Exception:
        return dict(tflops=1400.0, burst=1590.0, hbm=6650.0, source='fallback (B200_PROFILING.md)')


def host_threads():
    """CPU threads this process can really use: min(affinity mask, cgroup v2 cpu.max quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
        if quota != 'max':
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


# ------------------------------------------------------------------------------------------------------
# CPU arm: the oracle ports of the reference models (oracle/*.py, pinned to the reference at 1e-12), all host threads
# ------------------------------------------------------------------------------------------------------
def cpu_step_factory(workload, batch, forward_only=False):
    g = torch.Generator().manual_seed(1)
    frames = WORKLOADS[workload]['frames']
    if workload in ('timesformer', 'vivit'):
        from oracle import vt_oracle as O
        if workload == 'timesformer':
            cfg = dict(O.TIMESFORMER_B)
            sd = O.random_timesformer_state(cfg, seed=0)
            fwd = lambda x, training: O.timesformer_forward(sd, x, cfg, training=training)
        else:
            from videotransformer_pytorch_b200 import ViViT
            torch.manual_seed(0)
            m = ViViT(num_frames=16, img_size=IMG, patch_size=16, embed_dims=768, num_heads=12, num_transformer_layers=12)
            sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
            cfg = dict(num_frames_in=16, img_size=IMG, patch_size=16, embed_dims=768, num_heads=12, num_transformer_layers=12)
            fwd = lambda x, training: O.vivit_forward(sd, x, cfg, training=training)
        head_w = (torch.randn(NUM_CLASSES, 768, generator=g) * 0.02)
        head_b = torch.zeros(NUM_CLASSES)
        params = list(sd.values()) + [head_w, head_b]
        x = torch.randn(batch, frames, 3, IMG, IMG, generator=g)
        y = torch.randint(0, NUM_CLASSES, (batch,), generator=g)

        def loss_fn(training):
            return torch.nn.functional.cross_entropy(fwd(x, training) @ head_w.t() + head_b, y)
    else:
        from oracle import mvit_oracle as MO
        cfg = MO.maskfeat_config(img_size=IMG, num_frames=16, **{k: tuple(tuple(r) for r in v) if isinstance(v, list) else v
                                                                  for k, v in MASKFEAT_KW.items()})
        sd = MO.random_maskfeat_state(cfg, seed=0, dtype=torch.float32)
        params = list(sd.values())
        x = torch.randn(batch, frames, 3, IMG, IMG, generator=g)
        mask = (torch.rand(batch, 8, 14, 14, generator=g) < 0.4).float()
        target = torch.randn(batch, 16, 14, 14, 108, generator=g)
        markers = [[[0, 2], [5, 1]] for _ in range(batch)]
        if workload == 'mvit':
            loss_fn = lambda training: MO.maskfeat_forward_features(sd, x, None, cfg).square().mean()
        else:
            loss_fn = lambda training: MO.maskfeat_forward(sd, x, target, mask, markers, cfg)[1]

    if forward_only:          # BASELINE config 1: eval forward, no_grad
        def step():
            with torch.no_grad():
                return float(loss_fn(False))
        return step
    for v in params:
        v.requires_grad_(True)

    def step():
        for v in params:
            v.grad = None
        loss = loss_fn(True)
        loss.backward()
        return float(loss.detach())
    return step


def run_cpu(workload, steps, warmup, batch=1, forward_only=False):
    cores = host_threads()
    torch.set_num_threads(cores)
    step = cpu_step_factory(workload, batch, forward_only)
    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    total = sum(times)
    what = 'eval forward (no_grad)' if forward_only else 'fwd+bwd'
    return dict(value=batch * steps / total, ms_per_step=1e3 * total / steps, cores=cores,
                sample=f'{steps} timed step(s) of {what} on a {batch}-clip batch (fp32, torch CPU kernels, '
                       f'{cores} threads), {warmup} warm-up')


def main_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    # bounded: each step is a 1-clip sample of the per-GPU batch
    steps = max(1, min(args.steps, 8))
    warm = max(1, min(args.warmup, 2))
    r = run_cpu(args.workload, steps, warm, batch=1)
    f = run_cpu(args.workload, min(steps, 5), 1, batch=1, forward_only=True)
    line = {
        'metric': w['metric'], 'value': r['value'], 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps, 'warmup': warm,
        'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
        'config': {'workload': w['desc'], 'batch_per_gpu': 1, 'global_batch': 1, 'parallelism': 'cpu',
                   'arm': 'oracle PORT of the reference model on the host cores (fp32, torch CPU kernels; the reference is pure '
                          'Python and does not travel to the GPU box); each step is a 1-clip sample of the per-GPU batch'},
        'cpu_baseline': {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port', 'sample': r['sample'],
                         'forward_only': {'value': f['value'], 'unit': UNIT, 'ms_per_clip': f['ms_per_step'],
                                          'what': 'BASELINE config 1: single-clip eval forward, no_grad, fp32'}},
        'e2e': {'value': r['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(index), f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                       '-lms', '100'], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.f.read().splitlines():
            c = [v.strip() for v in ln.split(',')]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1])); pw.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': max(mx), 'power_w_max': max(pw), 'samples': len(sm),
                'reasons': sorted(reasons)}


class Trainee(torch.nn.Module):
    """TimeSformer-B + classification head, as built by the reference's VideoTransformer
    (model_trainer.py:53-82); loss = cross-entropy (training_step :204-206 without mixup)."""

    def __init__(self, arch='timesformer'):
        super().__init__()
        from videotransformer_pytorch_b200 import ClassificationHead, TimeSformer, ViViT
        if arch == 'timesformer':
            self.model = TimeSformer(num_frames=8, img_size=IMG, patch_size=16, embed_dims=768, num_heads=12,
                                     num_transformer_layers=12, attention_type='divided_space_time')
        else:
            self.model = ViViT(num_frames=16, img_size=IMG, patch_size=16, embed_dims=768, num_heads=12,
                               num_transformer_layers=12, attention_type='fact_encoder')
        self.cls_head = ClassificationHead(NUM_CLASSES, 768, eval_metrics='finetune')
        with torch.no_grad():   # temporal_fc is zero-init in the reference: make the branch live
            for n, p in self.model.named_parameters():
                if 'temporal_fc' in n:
                    p.normal_(std=0.02)

    def forward(self, x, y):
        return self.cls_head.loss(self.model(x), y)          # skinny-GEMV head + fused softmax-CE kernels


class MaskFeatStep(torch.nn.Module):
    """MaskFeat as built at model_trainer.py:54; `features_only` = BASELINE config 4 (the MViT-B backbone alone)."""

    def __init__(self, features_only):
        super().__init__()
        from videotransformer_pytorch_b200 import MaskFeat
        self.net = MaskFeat(**MASKFEAT_KW)
        self.features_only = features_only
        if features_only:       # backbone alone: the decoder and the mask token take no part (model_trainer.py:78-79 freezes the decoder)
            for p in self.net.decoder_pred.parameters():
                p.requires_grad = False
            self.net.mask_token.requires_grad = False

    def forward(self, x, target=None, mask=None, cmask=None):
        if self.features_only:
            return self.net.forward_features(x).square().mean()
        return self.net.forward_with_center_mask(x, target, mask, cmask)[1]


class WorkloadRun:
    """One workload on this rank: model, synthetic host batch, device-side input preparation."""

    def __init__(self, name, dev, B, rank):
        self.name, self.dev, self.B = name, dev, B
        self.w = WORKLOADS[name]
        g = torch.Generator().manual_seed(100 + rank)
        frames = self.w['frames']
        torch.manual_seed(0)
        if name in ('timesformer', 'vivit'):
            self.net = Trainee(name).to(dev).train()
            self.host = [torch.randn(B, frames, 3, IMG, IMG, generator=g).pin_memory(),
                         torch.randint(0, NUM_CLASSES, (B,), generator=g).pin_memory()]
            self.meta = None
        elif name == 'mvit':
            self.net = MaskFeatStep(True).to(dev).train()
            self.host = [torch.randn(B, frames, 3, IMG, IMG, generator=g).pin_memory()]
            self.meta = None
        else:
            from videotransformer_pytorch_b200.mask_generator import CubeMaskGenerator
            self.net = MaskFeatStep(False).to(dev).train()
            random.seed(rank)
            self.gen = CubeMaskGenerator((8, 14, 14), min_num_patches=16)
            self.host = [torch.randint(0, 256, (B, frames, IMG, IMG, 3), generator=g, dtype=torch.uint8).pin_memory(),
                         torch.zeros(B, 8, 14, 14).pin_memory()]
            self.meta = self.draw_masks()
        self.h2d_bytes = sum(t.numel() * t.element_size() for t in self.host)

    def draw_masks(self):
        """Per-sample cube masks on the host (reference data_trainer.py:28-31 / dataset.py:176-186), written into the pinned
        mask buffer; returns the [start, span] markers."""
        markers = []
        for i in range(self.B):
            m, cm = self.gen()
            self.host[1][i].copy_(torch.as_tensor(m, dtype=torch.float32))
            markers.append([[int(a), int(b)] for a, b in cm])
        return markers

    def prepare(self, dev_tensors, meta):
        """Device tensors as they arrive from the host -> the step's inputs (runs on the compute stream)."""
        if self.name != 'maskfeat':
            return tuple(dev_tensors)
        from videotransformer_pytorch_b200.hog import hog_targets_batch
        u8, mask = dev_tensors
        x = ((u8.float() * (1.0 / (255.0 * 0.225)) - 0.45 / 0.225)).permute(0, 1, 4, 2, 3).contiguous()   # ToTensor + Normalize
        target = hog_targets_batch(u8, meta)                      # dataset.py:188-196 on device, one launch for the batch
        cmask = self.net.net.center_frame_mask(mask, meta)
        return x, target, mask, cmask


def dump_outputs(net, loss, out_dir):
    """loss.npy and grad.<name>.npy for every parameter with a gradient; see --dump-outputs in the module docstring."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {'loss': loss.detach().reshape(1)}
    for n, p in net.named_parameters():
        if p.grad is None:
            continue
        g = p.grad.detach().reshape(-1)
        if g.numel() > DUMP_SAMPLE:
            idx = torch.randperm(g.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            g = g[idx.to(g.device)]
        arrays['grad.' + n] = g
    total = sum(a.numel() * (8 if a.dtype == torch.float64 else 4) for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f'--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte budget')
    for n, a in arrays.items():
        a = a.cpu()
        np.save(os.path.join(out_dir, n + '.npy'), a.numpy() if a.dtype == torch.float64 else a.float().numpy())
    return {'dir': out_dir, 'arrays': len(arrays), 'bytes': total}


def measure(run, args, world, rank, dist, steps, with_probe, dump_dir=None):
    """Times one workload: graph-captured step (value), e2e through host buffers, optional GEMM / attention probe;
    with dump_dir, writes the outputs of the last timed step there (dump_outputs)."""
    from videotransformer_pytorch_b200 import _lib
    from videotransformer_pytorch_b200.ddp import GradientBuckets
    from videotransformer_pytorch_b200.graph import GraphedTrainStep
    dev, net, B = run.dev, run.net, run.B
    reducer = GradientBuckets(net) if world > 1 else None
    dev_inputs = [t.to(dev) for t in run.host]
    step_inputs = run.prepare(dev_inputs, run.meta)

    def zero():
        if reducer is not None:
            reducer.zero_grad()
        else:
            for p in net.parameters():
                p.grad = None

    def eager_step(*inp):
        zero()
        loss = net(*inp)
        loss.backward()
        if reducer is not None:
            reducer.finish()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    step = eager_step
    graphed = None
    if not args.no_graph:
        # whole step (fwd + bwd [+ bucket all-reduces]) captured once, replayed with one launch per step
        graphed = GraphedTrainStep(net, step_inputs, reducer=reducer, warmup=3)
        step = lambda *inp: graphed(*inp)
    for _ in range(max(args.warmup, 3)):
        loss = step(*step_inputs)
    barrier()
    last = {}

    def timed_step():
        last['loss'] = step(*step_inputs)
    l0 = _lib.launch_count()
    ms_dev = timed(timed_step, steps)
    launches = (_lib.launch_count() - l0)
    if graphed is not None:      # replays launch the kernels recorded at capture time (the host-side counter is not touched)
        launches = graphed.kernels_per_replay * steps
    loss_value = float(loss.item())
    dumped = dump_outputs(net, last['loss'], dump_dir) if dump_dir else None

    # End to end through the public API: every step's batch comes from pinned host memory and the loss goes back to the
    # host.  The copy of step i+1 is issued on a copy stream while step i computes (double-buffered device staging),
    # exactly what a DataLoader with pin_memory + non_blocking transfers gives the reference's training loop.
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [[torch.empty_like(t) for t in dev_inputs] for _ in range(2)]
    arrived = [torch.cuda.Event(), torch.cuda.Event()]
    state = {'i': 0, 'meta': [run.meta, run.meta]}

    def issue_copy(slot):
        # no wait needed: the slot's previous consumer (two steps ago) finished before that step's loss.item() returned
        if run.name == 'maskfeat':
            state['meta'][slot] = run.draw_masks()                   # host-side mask generation is part of the step's input
        with torch.cuda.stream(copy_stream):
            for d, h in zip(bufs[slot], run.host):
                d.copy_(h, non_blocking=True)
            arrived[slot].record(copy_stream)
        if run.name == 'maskfeat':
            copy_stream.synchronize()                                # the pinned mask buffer is rewritten by the next draw

    def e2e_step():
        i = state['i']
        state['i'] = i + 1
        slot = i & 1
        torch.cuda.current_stream(dev).wait_event(arrived[slot])     # this step's input (host -> device) is here
        loss = step(*run.prepare(bufs[slot], state['meta'][slot]))
        issue_copy(slot ^ 1)                                         # next step's input travels during this step
        return float(loss.item())                                    # device -> host read of the loss

    issue_copy(0)
    e2e_step()
    ms_e2e = timed(e2e_step, steps)

    res = dict(ms_dev=ms_dev, ms_e2e=ms_e2e, launches=launches, loss=loss_value, dumped=dumped, reducer=reducer, graphed=graphed,
               step_inputs=step_inputs, eager_step=eager_step, kernels_per_replay=(graphed.kernels_per_replay if graphed else None))
    if with_probe:
        try:
            res['roofline'] = gemm_probe(run, args, reducer, step_inputs, eager_step, ms_dev / steps)
        except Exception as exc:             # the probe must never cost the headline line
            import traceback
            traceback.print_exc()
            pk = peaks()
            res['roofline'] = {'kernel': 'gemm_tcgen05_kernel / gemm2_tcgen05_kernel', 'bound': 'tensor', 'achieved': None,
                               'peak': pk['tflops'], 'unit': 'TFLOP/s', 'frac': None, 'traffic': None,
                               'error': f'{type(exc).__name__}: {str(exc)[:200]}',
                               'whole_step_frac_of_tensor_roofline':
                                   (run.w['flop_per_clip'] * run.B / (ms_dev / steps * 1e-3) / 1e12) / pk['tflops']}
    return res


def gemm_probe(run, args, reducer, step_inputs, eager_step, ms_per_step):
    """Roofline of the dominant kernel (the tcgen05 GEMMs), measured live: the SAME step captured once more with an external
    CUDA-event record node before and after every GEMM / attention launch on the capture stream; a replay yields the in-situ
    duration of each launch.  Launches carry a role tag (ops.py) so the attention-GEMM subset (qkv, QK^T, PV, out-proj:
    the north_star metric) is reported next to all GEMMs."""
    from videotransformer_pytorch_b200 import _lib
    from videotransformer_pytorch_b200.graph import GraphedTrainStep
    pk = peaks()
    rec = []
    K = _lib.K
    orig = {n: getattr(K, n) for n in ('gemm', 'attn_fwd', 'attn_bwd')}
    ext = {'external': True}

    def bracket(kind, flops, fn, *a, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True, **ext), torch.cuda.Event(enable_timing=True, **ext)
        e0.record()
        out = fn(*a, **kw)
        e1.record()
        rec.append((e0, e1, flops, kind))
        return out

    def timed_gemm(a, b, M, N, Kd, **kw):
        return bracket('gemm:' + str(kw.get('tag', '')), 2.0 * M * N * Kd, orig['gemm'], a, b, M, N, Kd, **kw)

    def timed_attn_fwd(qkv, Bp, N, H, hd, scale, **kw):
        return bracket('attn', 4.0 * Bp * H * N * N * hd, orig['attn_fwd'], qkv, Bp, N, H, hd, scale, **kw)

    def timed_attn_bwd(qkv, ctx, dctx, lse, Bp, N, H, hd, scale, **kw):
        return bracket('attn', 8.0 * Bp * H * N * N * hd, orig['attn_bwd'], qkv, ctx, dctx, lse, Bp, N, H, hd, scale, **kw)

    K.gemm, K.attn_fwd, K.attn_bwd = timed_gemm, timed_attn_fwd, timed_attn_bwd
    reps, timing = 1, None
    try:
        probe = None
        if not args.no_graph:
            try:
                rec.clear()
                probe = GraphedTrainStep(run.net, step_inputs, reducer=reducer, warmup=0)
            except Exception as exc:          # e.g. external events unsupported by this torch build
                sys.stderr.write(f'roofline: graph-event probe unavailable ({exc}); falling back to eager events\n')
                probe = None
        if probe is not None:
            for _ in range(2):
                probe(*step_inputs)
            torch.cuda.synchronize()
            timing = 'external CUDA-event nodes around every GEMM / attention launch inside the replayed step graph'
        else:
            ext.clear()
            rec.clear()
            reps = 2
            for _ in range(reps):
                torch.cuda._sleep(120_000_000)     # keeps the GPU busy while the host queues the step
                eager_step(*step_inputs)
            torch.cuda.synchronize()
            timing = 'CUDA events around every GEMM / attention launch of an eagerly issued step'
    finally:
        K.gemm, K.attn_fwd, K.attn_bwd = orig['gemm'], orig['attn_fwd'], orig['attn_bwd']
    gem = [(a.elapsed_time(b), f, k) for a, b, f, k in rec if k.startswith('gemm')]
    att = [(a.elapsed_time(b), f, k) for a, b, f, k in rec if k == 'attn']
    t_ms = sum(t for t, _, _ in gem)
    fl = sum(f for _, f, _ in gem)
    ach = fl / (t_ms * 1e-3) / 1e12
    # attention-GEMM subset: qkv + out-proj GEMMs (forward, dgrad, wgrad) and the attention cores
    sub = [(t, f) for t, f, k in gem if k in ('gemm:qkv', 'gemm:proj')] + [(t, f) for t, f, _ in att]
    sub_ms, sub_fl = sum(t for t, _ in sub), sum(f for _, f in sub)
    traffic = None
    try:
        with open(os.path.join(ROOT, 'profiles', 'gemm_traffic.json')) as fh:
            traffic = json.load(fh).get('dram_bytes_per_launch')
    except Exception:
        pass
    w = run.w
    roof = {'kernel': 'gemm_tcgen05_kernel / gemm2_tcgen05_kernel', 'bound': 'tensor', 'achieved': ach, 'peak': pk['tflops'],
            'unit': 'TFLOP/s', 'frac': ach / pk['tflops'], 'frac_of_burst': ach / pk['burst'], 'peak_burst': pk['burst'],
            'traffic': traffic, 'launches_timed': len(gem), 'gemm_ms_per_step': t_ms / reps, 'gemm_flop_per_step': fl / reps,
            'timing': timing, 'peak_source': pk['source'],
            'whole_step_frac_of_tensor_roofline': (w['flop_per_clip'] * run.B / (ms_per_step * 1e-3) / 1e12) / pk['tflops']}
    if sub_ms > 0:
        a2 = sub_fl / (sub_ms * 1e-3) / 1e12
        roof['attention_gemm'] = {
            'what': 'qkv + QK^T + PV + out-proj of the temporal and spatial passes, fwd+bwd (GEMM launches tagged qkv / proj + '
                    'attention-core kernels; algorithmic FLOPs, attention backward counted 2x forward)',
            'achieved': a2, 'frac': a2 / pk['tflops'], 'frac_of_burst': a2 / pk['burst'], 'ms_per_step': sub_ms / reps,
            'flop_per_step': sub_fl / reps, 'launches_timed': len(sub)}
    return roof


def gpu_eager_baseline(dev, B, steps=3):
    """SURVEY §8d's honest on-box comparator: the oracle port of the reference TimeSformer (the same torch ops the reference
    modules issue) in stock eager PyTorch on this GPU under bf16 autocast, same batch, fwd+bwd."""
    from oracle import vt_oracle as O
    cfg = dict(O.TIMESFORMER_B)
    sd = {k: v.to(dev).requires_grad_(True) for k, v in O.random_timesformer_state(cfg, seed=0).items()}
    g = torch.Generator().manual_seed(1)
    hw = (torch.randn(NUM_CLASSES, 768, generator=g) * 0.02).to(dev).requires_grad_(True)
    hb = torch.zeros(NUM_CLASSES, device=dev, requires_grad=True)
    x = torch.randn(B, 8, 3, IMG, IMG, generator=g).to(dev)
    y = torch.randint(0, NUM_CLASSES, (B,), generator=g).to(dev)

    def step():
        for v in list(sd.values()) + [hw, hb]:
            v.grad = None
        with torch.autocast('cuda', dtype=torch.bfloat16):
            feat = O.timesformer_forward(sd, x, cfg, training=True)
            loss = torch.nn.functional.cross_entropy(feat.float() @ hw.t() + hb, y)
        loss.backward()
        return loss

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {'value': B / (ms * 1e-3), 'unit': UNIT, 'ms_per_step': ms, 'steps': steps,
            'what': 'oracle port of the reference TimeSformer-B in stock eager PyTorch (ATen / cuBLAS kernels) under '
                    'torch.autocast(bfloat16) on this GPU, same batch, fwd+bwd'}


def ddp_check(run, res, dist):
    """N > 1: the bucketed mean the captured step leaves in p.grad vs the ranks' local gradients all-reduced eagerly."""
    net, dev = run.net, run.dev
    params = [p for p in net.parameters() if p.requires_grad]
    step_inputs = res['step_inputs']
    torch.manual_seed(4321)                         # same DropPath draws for both passes
    if res['graphed'] is not None:
        res['graphed'](*step_inputs)
    else:
        res['eager_step'](*step_inputs)
    torch.cuda.synchronize()
    got = torch.cat([p.grad.detach().reshape(-1) for p in params])
    torch.manual_seed(4321)
    loss = net(*step_inputs)
    local = torch.autograd.grad(loss, params)       # plain local gradients: no bucket hooks involved
    flat = torch.cat([g.reshape(-1) for g in local])
    dist.all_reduce(flat, op=dist.ReduceOp.AVG)
    num = (got - flat).norm()
    den = flat.norm()
    err = torch.stack([num / (den + 1e-30), (got - flat).abs().max() / (flat.abs().max() + 1e-30)])
    dist.all_reduce(err, op=dist.ReduceOp.MAX)
    return {'rel_l2': float(err[0]), 'max_rel_err': float(err[1]), 'elements': int(flat.numel()),
            'what': 'gradients left in the flat buckets by the captured step vs torch.autograd.grad of the same step '
                    'all-reduced (AVG) eagerly, same DropPath seed; max over ranks'}


def main_gpu(args):
    import torch.distributed as dist
    from videotransformer_pytorch_b200 import _lib

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the hot path has no CPU fallback; use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        import datetime
        dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=300))
    _lib.load_library()
    if world > 1 and args.reserve_sms:
        _lib.set_reserved_sms(args.reserve_sms)      # room for the overlapped NCCL all-reduce kernels

    name = args.workload
    w = WORKLOADS[name]
    B = args.batch or w['batch']
    run = WorkloadRun(name, dev, B, rank)
    sampler = ClockSampler(torch.cuda.current_device()) if rank == 0 else None
    res = measure(run, args, world, rank, dist, args.steps, with_probe=True,
                  dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop() if sampler else None
    check = None
    if world > 1:
        try:
            check = ddp_check(run, res, dist)
        except Exception as exc:
            import traceback
            traceback.print_exc()
            check = {'error': f'{type(exc).__name__}: {str(exc)[:200]}'}

    exposed = None
    if world > 1 and not args.no_graph:
        # the same step without the exchange (local gradients only) on every rank: what the all-reduce adds to the step
        from videotransformer_pytorch_b200.graph import GraphedTrainStep
        try:
            solo = GraphedTrainStep(run.net, res['step_inputs'], reducer=None, warmup=0)
            for _ in range(3):
                solo(*res['step_inputs'])
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                solo(*res['step_inputs'])
            e1.record()
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            exposed = {'allreduce_exposed_ms': res['ms_dev'] / args.steps - float(t), 'ms_per_step_without_exchange': float(t)}
            del solo
        except Exception as exc:
            exposed = {'error': str(exc)[:200]}

    others = {}
    if args.others and name == 'timesformer' and args.batch == 0:
        del res['graphed']
        for other in ('vivit', 'mvit', 'maskfeat'):
            try:
                torch.cuda.empty_cache()
                r2 = WorkloadRun(other, dev, WORKLOADS[other]['batch'], rank)
                k = max(3, min(args.steps, 5))
                m = measure(r2, args, world, rank, dist, k, with_probe=False)
                pk = peaks()
                ms = m['ms_dev'] / k
                others[other] = {
                    'workload': WORKLOADS[other]['desc'], 'batch_per_gpu': r2.B, 'steps': k,
                    'value': world * r2.B / (ms * 1e-3), 'unit': UNIT, 'ms_per_step': ms,
                    'e2e': {'value': world * r2.B * k / (m['ms_e2e'] * 1e-3), 'ms_per_step': m['ms_e2e'] / k,
                            'h2d_bytes_per_step': r2.h2d_bytes, 'd2h_bytes_per_step': 4},
                    'kernels_per_replay': m['kernels_per_replay'], 'loss': m['loss'],
                    'whole_step_frac_of_tensor_roofline': (WORKLOADS[other]['flop_per_clip'] * r2.B / (ms * 1e-3) / 1e12) / pk['tflops'],
                }
                del m, r2
            except Exception as exc:
                import traceback
                traceback.print_exc()
                others[other] = {'error': f'{type(exc).__name__}: {str(exc)[:300]}'}

    if world > 1:
        dist.barrier()
    cpu = cpu_fwd = eager = None
    if rank == 0:
        k_cpu = 5 if args.baselines else 1
        cpu = run_cpu(name, steps=k_cpu, warmup=1 if args.baselines else 0, batch=1)
        cpu_fwd = run_cpu(name, steps=k_cpu, warmup=1 if args.baselines else 0, batch=1, forward_only=True)
        if name == 'timesformer' and world == 1 and args.baselines:
            try:
                eager = gpu_eager_baseline(dev, B)
            except Exception as exc:
                eager = {'error': f'{type(exc).__name__}: {str(exc)[:200]}'}
    if rank == 0:
        steps = args.steps
        value = world * B * steps / (res['ms_dev'] * 1e-3)
        e2e = world * B * steps / (res['ms_e2e'] * 1e-3)
        roof = res['roofline']
        line = {
            'metric': w['metric'], 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': res['ms_dev'] / steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': w['desc'], 'batch_per_gpu': B, 'global_batch': B * world,
                       'parallelism': f'dp{world}', 'residual_stream': 'fp32', 'gemm_operands': 'bf16/fp32-accum',
                       'optimizer': 'excluded (metric is fwd+bwd)',
                       'launch': 'eager' if args.no_graph else 'cuda-graph replay (fwd+bwd captured once)',
                       'grad_allreduce': f'fp32 buckets, NCCL AVG, overlapped with backward inside the graph, {args.reserve_sms} SMs reserved' if world > 1 else 'n/a',
                       'l2': 'per-step working set ~5 GB >> 126 MB L2 (no flush needed)',
                       'parity_gate': 'per-block 1e-3 rel (fp32 residual stream); end to end vs the fp64 oracle at this very shape '
                                      '(tests/test_gpu_baseline_shapes.py): feature 7e-3, gradients <= 1.1e-2 — below the reference\'s own '
                                      'bf16-autocast error (9e-3 / 1.3e-2)'},
            'e2e': {'value': e2e, 'unit': UNIT, 'ms_per_step': res['ms_e2e'] / steps,
                    'h2d_bytes_per_step': run.h2d_bytes, 'd2h_bytes_per_step': 4},
            'gpu_launches': res['launches'], 'kernels_per_replay': res['kernels_per_replay'], 'loss': res['loss'],
            'clocks': clocks, 'roofline': roof,
            'cpu_baseline': {'value': cpu['value'], 'unit': UNIT, 'cores': cpu['cores'], 'kind': 'port', 'sample': cpu['sample'],
                             'forward_only': {'value': cpu_fwd['value'], 'unit': UNIT, 'ms_per_clip': cpu_fwd['ms_per_step'],
                                              'what': 'BASELINE config 1: single-clip eval forward, no_grad, fp32'}},
        }
        if eager is not None:
            line['gpu_eager_baseline'] = eager
        if check is not None:
            line['ddp_check'] = check
        if exposed is not None:
            line['exchange'] = exposed
        if others:
            line['other_workloads'] = others
        if res['dumped'] is not None:
            line['dumped_outputs'] = res['dumped']
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        # captured graphs hold NCCL kernels: release them before the communicator goes away
        res = run = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default='timesformer', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=0, help='clips per GPU (0 = the BASELINE config: 8, maskfeat 16)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--reserve-sms', type=int, default=0, help='SMs kept free of persistent GEMM CTAs when N > 1 (NCCL overlap)')
    ap.add_argument('--no-graph', action='store_true', help='issue the step kernel by kernel instead of replaying a CUDA graph')
    ap.add_argument('--no-others', dest='others', action='store_false', help='skip the other BASELINE configs in the default line')
    ap.add_argument('--no-baselines', dest='baselines', action='store_false', help='skip the CPU / eager-GPU comparators (A/B runs)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the loss and parameter gradients of the last timed step '
                                                          'to DIR/<name>.npy (gradients sampled: see the module docstring)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return main_reference(args)
    if int(os.environ.get('WORLD_SIZE', '1')) > 1 or args.workload != 'timesformer':
        return main_gpu(args)
    try:
        return main_gpu(args)
    except SystemExit:
        raise
    except Exception as exc:
        # One GPU, default workload: never lose the headline line to a bug in the newer measurement code — re-run the copy of
        # this benchmark that was confirmed on hardware (tools/bench_v1.py) in a fresh process (fresh CUDA context).
        import traceback
        traceback.print_exc()
        sys.stderr.write(f'bench.py: measurement raised {type(exc).__name__}; falling back to tools/bench_v1.py\n')
        cmd = [sys.executable, os.path.join(ROOT, 'tools', 'bench_v1.py'), '--gpus', '1', '--steps', str(args.steps),
               '--warmup', str(args.warmup)] + (['--no-graph'] if args.no_graph else [])
        out = subprocess.run(cmd, capture_output=True, text=True)
        sys.stderr.write(out.stderr[-4000:])
        lines = [ln for ln in out.stdout.splitlines() if ln.startswith('{')]
        if not lines:
            raise
        line = json.loads(lines[-1])
        line['fallback'] = f'tools/bench_v1.py after {type(exc).__name__}: {str(exc)[:160]}'
        print(json.dumps(line), flush=True)


if __name__ == '__main__':
    main()
