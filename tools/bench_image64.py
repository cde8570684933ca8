"""GPU: the 3x64x64 sweep -- teacher (sf 1.0) against the sf 0.5 student, 50 steps, 8 guidance scales, fp16 -- as one JSON line.

    python tools/bench_image64.py [seeds per chunk (512)] [--out FILE]

Reports, all read in this one run:
  * trajectories/s of the device-resident chunk (grid.run_chunk on a pre-staged chunk, CUDA events; one untimed chunk first)
    and of grid.sweep end to end (host draws, uploads, samplers, metrics, read-back; wall clock after a device synchronise);
  * conv TFLOP/s: the samplers' executed conv flops (real channels, taps that meet the map) over the device-resident chunk time,
    and over the conv kernels' own time in one profiled (event per launch) pass;
  * peak device memory (torch.cuda.max_memory_allocated) of one sweep at the default chunk in fp16 and in TF32, and the chunk
    grid.sweep chose;
  * an A/B of the 32x32-level layer shapes (enc2 / dec1 of the 64x64 models) in the generic [image][y][x] tiles against the
    halo form, kernel-only (dtraj_bench_conv, zero-filled operands, 20 launches between one event pair) at the sweep's rows,
    conv2 with its fused 1x1 residual conv;
  * the GPU name and power limit (nvidia-smi)."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from distillation_trajectories_b200 import _lib, grid
from distillation_trajectories_b200.engine import UNetEngine


class Cfg64(bench.Cfg):          # 3x64x64, 50 steps
    channels, image_size = 3, 64


# the 32x32-level layers of a 64x64 model with first-block width b and width m: (name, c0, c1, cout, ksize, flags); conv2 carries the
# block's 1x1 residual conv as extra MMAs (CONV_RESACC = 128: c1 = its input channels), as in the forward
def AB_LAYERS(b, m):
    return (("enc2.conv1", b, 0, m, 3, 1), ("enc2.conv2", m, b, m, 3, 1 | 128),
            ("dec1.conv1", m, m, b, 3, 1), ("dec1.conv2", b, 2 * m, b, 3, 1 | 128))


def layer_flops(n, c0, c1, cout, flags):
    if flags & 128:
        return 2.0 * n * 32 * 32 * cout * (c0 * 9 + c1)
    return 2.0 * n * 32 * 32 * cout * (c0 + c1) * 9


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, clk = [c.strip() for c in out.split(",")]
        return {"gpu": name, "power_limit": plim, "sm_clock_max": clk}
    except Exception as e:             # (reported, not guessed)
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_file = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out_file in args:
        args.remove(out_file)
    S = int(args[0]) if args else 512
    dev = torch.device("cuda", 0)
    cfg, G = Cfg64, bench.GUIDANCE
    teacher = bench.make_model(cfg, 1.0, 0, dev)
    student = bench.make_model(cfg, 0.5, 1050, dev)
    res = {"workload": f"3x64x64, teacher sf 1.0 vs student sf 0.5, {cfg.timesteps} steps, CFG w in {G}, sampler S2 + pair metrics, f16",
           "seeds_per_chunk": S, "pairs_per_chunk": S * len(G)}
    res.update(gpu_info())

    # device-resident chunk: one untimed (builds, captures), one timed
    chunks = [grid.stage_chunk(list(range(i * S, (i + 1) * S)), cfg, G, dev) for i in range(2)]
    torch.cuda.synchronize()
    grid.run_chunk(teacher, [student], chunks[0], dev, "f16")
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _, _, n_traj = grid.run_chunk(teacher, [student], chunks[1], dev, "f16")
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    res["device_resident"] = {"trajectories": n_traj, "ms": round(ms, 1), "trajectories_per_s": round(n_traj / ms * 1e3, 1)}
    samplers = bench.samplers_of([teacher, student], cfg, "f16", dev)
    fl = sum(sum(s.flops()) for s in samplers)
    prof = [s.profile() for s in samplers]
    conv_ms = sum(p["ms"][0] + p["ms"][4] for p in prof)
    res["conv"] = {"executed_tflop_per_chunk": round(fl / 1e12, 2),
                   "tflops_over_chunk_time": round(fl / (ms / 1e3) / 1e12, 1),
                   "tflops_over_conv_kernel_time": round(fl / (conv_ms / 1e3) / 1e12, 1),
                   "note": "executed flops: real channels, taps that meet the map, fused enc1 conv2 included; conv kernel time from "
                           "one pass with an event pair around every launch"}
    rows = [s.n_rows for s in samplers]
    del chunks, samplers, prof            # (a closed sampler's buffers live as long as the Python object)
    bench.close_engines([teacher, student])
    torch.cuda.empty_cache()

    # end to end and peak memory at the default chunk (max_pairs = 4096), fp16 and TF32
    mem = {}
    for prec in ("f16", "tf32"):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        st = {}
        t0 = time.perf_counter()
        grid.sweep(teacher, {"s": student}, cfg, G, S, dev, precision=prec, reduce=False, stats=st)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        chunk = grid.seeds_per_chunk_64(teacher, [student], cfg, len(G), prec, dev)
        mem[prec] = {"peak_gb": round(torch.cuda.max_memory_allocated(dev) / 1e9, 2), "seeds_per_chunk": min(chunk, 4096 // len(G))}
        if prec == "f16":        # (the first sweep also builds and captures the loops of its chunk shape: timed again below)
            t0 = time.perf_counter()
            grid.sweep(teacher, {"s": student}, cfg, G, S, dev, precision=prec, reduce=False, stats=st)
            torch.cuda.synchronize()
            sec = time.perf_counter() - t0
            res["end_to_end"] = {"seeds": S, "trajectories": 2 * S * len(G), "s": round(sec, 3),
                                 "trajectories_per_s": round(2 * S * len(G) / sec, 1)}
        bench.close_engines([teacher, student])
        torch.cuda.empty_cache()
    res["memory"] = mem

    # A/B of the 32x32-level layers: generic tiles (debug = 2) against the halo form (debug = 0), kernel only
    lib = _lib.load()
    ab = []
    for tag, b, m, n in (("teacher", 128, 256, rows[0]), ("student0.5", 64, 128, rows[1])):
        for name, c0, c1, cout, k, flags in AB_LAYERS(b, m):
            flops = layer_flops(n, c0, c1, cout, flags)
            r = {"model": tag, "layer": name, "rows": n}
            for form, dbg in (("generic", 2), ("halo", 0)):
                t = C.c_float()
                _lib.check(lib.dtraj_bench_conv(_lib.PREC_F16, c0, c1, cout, n, 32, k, flags, 20, dbg, C.byref(t)))
                r[form + "_us"] = round(t.value * 1e3, 1)
                r[form + "_tflops"] = round(flops / (t.value / 1e3) / 1e12, 1)
            ab.append(r)
    res["ab_32x32_generic_vs_halo"] = ab
    res["umma_error"] = int(lib.dtraj_debug_umma_error())
    line = json.dumps(res)
    print(line)
    if out_file:
        with open(out_file, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
