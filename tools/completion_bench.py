"""Throughput of scene-graph completion against unconditioned sampling on one GPU.

    python tools/completion_bench.py --out DIR [--batch 512] [--num-steps 256] [--repeats 2]

Workload: the Visual Genome geometry, batch 512, 256 sampler steps, CUDA graphs and padding skipping on (the sampler
defaults), the node counts of bench.py.  Completion condition: half of the valid nodes with class and box known, plus
every relation among the known nodes (object completion).  After one warm-up call of each, unconditioned
``sample_on_device`` and ``sample_completion`` alternate, ``--repeats`` times each, in this one process, so both see the
same clocks; each call is timed by a host clock around work that ends in a device synchronise.  The card's name, power
limit and SM clocks are read (read-only ``nvidia-smi`` queries) before and after the timed calls.  Writes
DIR/completion_bench.json and prints it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from diffusesg_b200 import native  # noqa: E402
from diffusesg_b200.model.diffusesg.diffusesg import DiffuseSG  # noqa: E402
from diffusesg_b200.model.precond.precond import NodeAdjPrecond  # noqa: E402
from diffusesg_b200.runner.mcmc_sampler import completion  # noqa: E402
from diffusesg_b200.runner.mcmc_sampler.edm import NodeAdjEDMSampler  # noqa: E402
from diffusesg_b200.utils.synthetic import CONFIGS, in_chans, synthetic_node_flags, synthetic_state_dict  # noqa: E402

NUM_ADJ_TYPE, NUM_NODE_TYPE = 51, 150   # Visual Genome


def gpu_info(index: int) -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))


def condition(flags: torch.Tensor, seed: int):
    g = torch.Generator().manual_seed(seed)
    b, n = flags.shape
    pick = flags & (torch.rand(b, n, generator=g) < 0.5)
    node_cls = torch.where(pick, torch.randint(0, NUM_NODE_TYPE, (b, n), generator=g), torch.full((b, n), -1))
    bbox = torch.where(pick[..., None], torch.rand(b, n, 4, generator=g), torch.full((b, n, 4), float("nan")))
    pair = pick[:, :, None] & pick[:, None, :] & ~torch.eye(n, dtype=torch.bool)
    adj_cls = torch.where(pair, torch.randint(0, NUM_ADJ_TYPE, (b, n, n), generator=g), torch.full((b, n, n), -1))
    return node_cls, bbox, adj_cls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--num-steps", type=int, default=256)
    ap.add_argument("--repeats", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("completion_bench.py: no CUDA device (the native path has no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    native.lib()
    cfg = CONFIGS["vg"]
    B, N, ce, cn = args.batch, cfg["img"], cfg["c_e"], cfg["c_n"]
    torch.manual_seed(1234)
    np.random.seed(1234)
    net = DiffuseSG(img_size=N, in_chans=in_chans(cfg), patch_size=1, embed_dim=cfg["embed"], depths=cfg["depths"],
                    num_heads=[3, 6, 12, 24], window_size=cfg["window"], mlp_ratio=4., drop_rate=0., attn_drop_rate=0.,
                    drop_path_rate=0.0, self_condition=cfg["self_cond"], symmetric_noise=False, out_chans_adj=ce,
                    out_chans_node=cn)
    net.load_state_dict(synthetic_state_dict(cfg, seed=1234, stress=False), strict=True)
    model = NodeAdjPrecond(precond="edm", model=net.to(dev), self_condition=cfg["self_cond"],
                           symmetric_noise=False).eval()
    sampler = NodeAdjEDMSampler(num_steps=args.num_steps, clip_samples=True, clip_samples_min=-1.0,
                                clip_samples_max=1.0, clip_samples_scope="x_0", dev=dev, objective="edm",
                                self_condition=cfg["self_cond"], symmetric_noise=False)
    flags_host = synthetic_node_flags(cfg, B, seed=1234)
    flags = flags_host.to(dev)
    known = completion.encode_known(flags, ce, cn, *condition(flags_host, 99), NUM_ADJ_TYPE, NUM_NODE_TYPE)
    init = (torch.randn(B, ce, N, N, device=dev), torch.randn(B, N, cn, device=dev))
    n_known = dict(nodes=int((~known[1][..., 0].isnan()).sum()), relations=int((~known[0][:, 0].isnan()).sum()),
                   valid_nodes=int(flags.sum()))

    def unconditioned():
        sampler.sample_on_device(model, flags, init_adjs=init[0], init_nodes=init[1], num_node_chan=cn, num_edge_chan=ce)

    def completed():
        sampler.sample_completion(model, flags, *known, init_adjs=init[0], init_nodes=init[1], num_node_chan=cn,
                                  num_edge_chan=ce)

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    unconditioned()
    completed()
    before = gpu_info(0)
    runs = []
    for r in range(args.repeats):
        for kind, fn in (("sample_on_device", unconditioned), ("sample_completion", completed)):
            s = timed(fn)
            runs.append(dict(kind=kind, repeat=r, seconds=s, graphs_per_s=B / s))
    after = gpu_info(0)
    rate = lambda k: [x["graphs_per_s"] for x in runs if x["kind"] == k]
    u, c = rate("sample_on_device"), rate("sample_completion")
    result = dict(workload=dict(config="vg", batch=B, num_steps=args.num_steps, graphs=sampler.use_graphs,
                                padding_skipping=sampler.skip_padding, condition=n_known),
                  gpu_before=before, gpu_after=after, runs=runs,
                  mean_graphs_per_s=dict(sample_on_device=float(np.mean(u)), sample_completion=float(np.mean(c))),
                  completion_overhead_pct=float(100.0 * (np.mean(u) / np.mean(c) - 1.0)))
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "completion_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
