"""Time the 16 x 16-window attention backward (dsg_tr_window_attention_bwd_w16) on the five shapes of n64w16.

    python tools/attention_bwd_w16_bench.py --out DIR [--batch 128] [--launches 50] [--rounds 3]

Shapes (res, shift, heads): the 16 x 16-window blocks of the n64w16 geometry (depths [2, 2, 6, 2]): res 64 with 3 heads
and res 32 with 6 heads, each unshifted and shifted by 8, and res 16 (one window per sample) with 12 heads.  Per shape:
five warm-up launches, then `--rounds` windows of `--launches` back-to-back launches between two CUDA events; the median
window gives the time per launch.  At batch 128 each shape's q / k / v / dO / dqkv (75-300 MB) exceeds the 126 MB L2.
Rates come from the shapes, per window-head: five 256 x 256 x 32 products (21.0 MFLOP), 65,536 exponentials and the
HBM traffic of reading q, k, v, dO and writing dq, dk, dv once (7 x 256 x 32 bf16 = 112 KiB).  The per-iteration total
weights each shape by its number of blocks in one backward pass (2, 2, 2, 2 and 12: 432 window-heads per sample).
The card's name and power limit are read (read-only nvidia-smi query) in the same process.  Writes
DIR/attention_bwd_w16_bench.json and prints it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from diffusesg_b200 import native  # noqa: E402

# (res, shift, heads, blocks of that shape in one n64w16 backward pass)
SHAPES = [(64, 0, 3, 2), (64, 8, 3, 2), (32, 0, 6, 2), (32, 8, 6, 2), (16, 0, 12, 12)]
FLOP_PER_WH = 5 * 2 * 256 * 256 * 32
EXP_PER_WH = 256 * 256
BYTES_PER_WH = 7 * 256 * 32 * 2


def gpu_info(index: int) -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))


def time_shape(batch: int, res: int, shift: int, heads: int, launches: int, rounds: int, dev) -> float:
    c = heads * 32
    g = torch.Generator(device=dev).manual_seed(res + shift + heads)
    qkv = (torch.randn(batch * res * res, 3 * c, device=dev, generator=g) * 0.5).to(torch.bfloat16)
    datt = torch.randn(batch * res * res, c, device=dev, generator=g).to(torch.bfloat16)
    table = torch.randn(31 * 31, heads, device=dev, generator=g) * 0.5
    dqkv = torch.empty_like(qkv)
    dtable = torch.zeros_like(table)
    lib, st = native.lib(), native.stream_ptr(dev)

    def launch():
        native.check(lib.dsg_tr_window_attention_bwd_w16(qkv.data_ptr(), datt.data_ptr(), table.data_ptr(), dqkv.data_ptr(),
                                                         dtable.data_ptr(), batch, res, 16, shift, heads, st), "bwd_w16")
    for _ in range(5):
        launch()
    torch.cuda.synchronize(dev)
    times = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            launch()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / launches)
    if not torch.isfinite(dqkv.float()).all():
        raise RuntimeError(f"non-finite gradient at res {res} shift {shift} heads {heads}")
    return sorted(times)[len(times) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_bwd_w16_bench: no CUDA device (this measures the B200 kernel; there is no CPU path)")
    dev = torch.device("cuda:0")
    info = gpu_info(0)
    rows = []
    iter_ms = iter_wh = 0.0
    for res, shift, heads, blocks in SHAPES:
        ms = time_shape(a.batch, res, shift, heads, a.launches, a.rounds, dev)
        wh = a.batch * (res // 16) ** 2 * heads
        rows.append(dict(res=res, shift=shift, heads=heads, blocks_per_pass=blocks, window_heads=wh, ms=round(ms, 4),
                         tflops=round(wh * FLOP_PER_WH / ms / 1e9, 1), gbps=round(wh * BYTES_PER_WH / ms / 1e6, 1),
                         gexp_per_s=round(wh * EXP_PER_WH / ms / 1e6, 1)))
        iter_ms += blocks * ms
        iter_wh += blocks * wh
    out = dict(gpu=info, batch=a.batch, launches=a.launches, rounds=a.rounds, shapes=rows,
               per_iteration=dict(window_heads=int(iter_wh), ms=round(iter_ms, 3),
                                  tflop=round(iter_wh * FLOP_PER_WH / 1e12, 3), gb=round(iter_wh * BYTES_PER_WH / 1e9, 2),
                                  tflops=round(iter_wh * FLOP_PER_WH / iter_ms / 1e9, 1),
                                  gbps=round(iter_wh * BYTES_PER_WH / iter_ms / 1e6, 1)))
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "attention_bwd_w16_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
