"""How much error does the REFERENCE algorithm itself show under bf16 autocast at the BASELINE shapes?

Runs the oracle port (pinned to the reference at 1e-12) of TimeSformer-B / ViViT-B on the CPU twice — fp64 and fp32
under torch.autocast(bfloat16) — in train mode with the same DropPath seed, and prints the rel-L2 error of the cls
feature, the loss and every parameter gradient.  The constants gate tests/test_gpu_baseline_shapes.py
(SURVEY.md §8c: "no worse than 1.5x the reference-bf16-autocast error").

    python tools/ref_autocast_error.py [timesformer|vivit] [B] [input size]

The input size (default 224) is the clip's height and width; the models stay built at 224, so for TimeSformer another
size runs through the bicubic pos_embed interpolation (448: the 785-token frames of high-resolution fine-tuning).
"""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import interp_oracle as IO   # noqa: E402
from oracle import vt_oracle as O   # noqa: E402


def rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else 'timesformer'
    B = int(sys.argv[2]) if len(sys.argv) > 2 else 2
    S = int(sys.argv[3]) if len(sys.argv) > 3 else 224
    torch.set_num_threads(os.cpu_count())
    g = torch.Generator().manual_seed(1)
    if which == 'timesformer':
        cfg = dict(O.TIMESFORMER_B)
        sd = O.random_timesformer_state(cfg, seed=0)
        x = torch.randn(B, 8, 3, S, S, generator=g)
        fwd = lambda s, xx: IO.forward(s, xx, cfg, 'divided_space_time', training=True)
    else:
        from tests.test_gpu_baseline_shapes import vivit_b_state
        cfg, sd = vivit_b_state()
        x = torch.randn(B, 16, 3, S, S, generator=g)
        fwd = lambda s, xx: O.vivit_forward(s, xx, cfg, training=True)
    hw = torch.randn(400, 768, generator=g) * 0.02
    y = torch.randint(0, 400, (B,), generator=g)

    def run(dtype, autocast):
        s = {k: v.detach().clone().to(dtype).requires_grad_(True) for k, v in sd.items()}
        torch.manual_seed(7)
        t0 = time.time()
        with torch.autocast('cpu', dtype=torch.bfloat16, enabled=autocast):
            f = fwd(s, x.to(dtype))
            loss = torch.nn.functional.cross_entropy(f.float() @ hw.to(f.dtype).float().t() if autocast else f @ hw.to(dtype).t(), y)
        loss.backward()
        print(f'  {dtype} autocast={autocast}: {time.time() - t0:.1f}s', flush=True)
        return f.detach(), float(loss.detach()), {k: v.grad for k, v in s.items()}

    f64, l64, g64 = run(torch.float64, False)
    f32, l32, g32 = run(torch.float32, False)
    fac, lac, gac = run(torch.float32, True)
    print(f'{which} B={B} {S}x{S}: fp32 vs fp64: feature {rel(f32, f64):.2e} loss {abs(l32 - l64) / abs(l64):.2e}')
    print(f'{which} B={B} {S}x{S}: bf16-autocast vs fp64: feature {rel(fac, f64):.2e} loss {abs(lac - l64) / abs(l64):.2e}')
    errs = sorted(((rel(gac[k], g64[k]), k) for k in g64), reverse=True)
    e32 = max(rel(g32[k], g64[k]) for k in g64)
    print(f'grads: fp32 worst {e32:.2e}; autocast worst {errs[0][0]:.2e} ({errs[0][1]}), median {errs[len(errs) // 2][0]:.2e}')
    for e, k in errs[:8]:
        print(f'   {e:.2e} {k}')


if __name__ == '__main__':
    main()
