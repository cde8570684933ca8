"""GPU: per-launch device time of ONE forward + step of a captured S2 loop, for any image size / student width.

    python tools/profile_layers.py <H: 16|32|64> <seeds> <size factors, comma separated> [precision] [w]

Every (seed, w) pair of a model is one sample (CFG: two forward rows).  Uses dtraj_sampler_profile_text: the loop runs
un-captured with a CUDA event pair around every launch, the table is the SECOND step's launches (warm caches, real data).
Prints per layer: grid, microseconds, algorithmic TFLOP/s, and the model's totals."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from distillation_trajectories_b200 import grid
from distillation_trajectories_b200.engine import UNetEngine

H = int(sys.argv[1]) if len(sys.argv) > 1 else 16
seeds = int(sys.argv[2]) if len(sys.argv) > 2 else 296
sfs = [float(a) for a in sys.argv[3].split(",")] if len(sys.argv) > 3 else [1.0, 0.5]
prec = sys.argv[4] if len(sys.argv) > 4 else "f16"
scales = [float(sys.argv[5])] if len(sys.argv) > 5 else (bench.GUIDANCE if H == 16 else [7.5])


class Cfg64(bench.Cfg):          # 3x64x64, 50 steps (the bench configs stop at 32x32)
    channels, image_size = 3, 64


cfg = {16: bench.Cfg, 32: bench.Cfg32, 64: Cfg64}[H]
dev = torch.device("cuda", 0)
ck = grid.stage_chunk(list(range(seeds)), cfg, scales, dev)
print(f"# {cfg.channels}x{H}x{H}, {seeds} seeds x {len(scales)} scales, precision {prec}; second step of the loop, CUDA events per launch")
for sf in sfs:
    m = bench.make_model(cfg, sf, 0 if sf == 1.0 else 1000 + int(sf * 100), dev)
    grid.run_chunk(m, [m], ck, dev, prec)
    torch.cuda.synchronize()
    s = next(reversed(UNetEngine.for_model(m, H, cfg.timesteps, prec, dev)._samplers.values()))
    s.profile_layers(1)
    rows = s.profile_layers(1)
    tot_us, tot_fl = sum(r[2] for r in rows), sum(r[3] for r in rows)
    print(f"== sf={sf} dims={m.dims} forward rows={s.n_rows}: {tot_us:.0f} us per forward+step, {tot_fl / tot_us / 1e6:.0f} TFLOP/s algorithmic")
    print(f"{'layer':38s} {'grid':>5s} {'us':>8s} {'TF/s':>7s} {'share':>6s}")
    for name, g, us, fl in rows:
        print(f"{name:38s} {g:5d} {us:8.1f} {fl / us / 1e6 if fl else 0:7.0f} {us / tot_us * 100:5.1f}%")
    UNetEngine.invalidate(m)
    del m, s
    torch.cuda.empty_cache()
