"""GPU: the shared-memory split of the 32x32-level halo layers (enc2 / dec1 of 3x64x64 models), kernel only.

    python tools/halo_split_ab.py [rows (7680)]

For each layer of the teacher (sf 1.0) and the sf 0.5 student: microseconds (dtraj_bench_conv, zero-filled operands, 20 launches
between one event pair) of the split build_umma_launch chooses and of every (halo slots, epilogue buffers per warp) pair, the
rest of the shared memory going to weight stages.  Prints the GPU name and power limit first."""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_image64 import AB_LAYERS, layer_flops
from distillation_trajectories_b200 import _lib

rows = int(sys.argv[1]) if len(sys.argv) > 1 else 7680
lib = _lib.load()
print("#", subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip())
splits = [(h, e) for h in (2, 3, 4) for e in (1, 2)]
print(f"# {rows} rows of 32x32, fp16; us per launch (TFLOP/s); 'plan' = the split the forward uses")
print(f"{'model':10s} {'layer':11s} {'plan':>14s} " + " ".join(f"{'hb%d/epi%d' % s:>14s}" for s in splits))
for tag, b, m in (("teacher", 128, 256), ("sf0.5", 64, 128)):
    for name, c0, c1, cout, k, flags in AB_LAYERS(b, m):
        fl = layer_flops(rows, c0, c1, cout, flags)
        cells = []
        for dbg in [0] + [0x100 | h << 4 | e for h, e in splits]:
            t = C.c_float()
            rc = lib.dtraj_bench_conv(_lib.PREC_F16, c0, c1, cout, rows, 32, k, flags, 20, dbg, C.byref(t))
            cells.append(f"{t.value * 1e3:7.1f} ({fl / (t.value / 1e3) / 1e12:4.0f})" if rc == 0 else f"{'-':>14s}")
        print(f"{tag:10s} {name:11s} " + " ".join(f"{c:>14s}" for c in cells), flush=True)
print("umma_error", lib.dtraj_debug_umma_error())
