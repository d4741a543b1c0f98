"""Cost of reconstruction-guided completion (DESIGN.md §3.7) on one GPU.

    python tools/guided_completion_bench.py --out DIR [--batches 128,256,512,1024] [--num-steps 16] [--repeats 2]
                                            [--guidance 0.5]

Workload: the Visual Genome geometry with the node counts of bench.py, object completion (half of the valid nodes with
class and box known, plus every relation among them).  B = 128 first, then the larger batches in order until one does
not fit; the largest that ran is the "largest batch that fits" of the list.  Per batch, after one warm-up call of each:
  * unguided ``sample_completion`` (its default path: CUDA graphs, padding skipping) and guided ``sample_completion``
    (eager, dense), alternated ``--repeats`` times, each timed with CUDA events around the call: ms per sampler step;
  * the denoiser backward of one preconditioned call (coin off), timed with CUDA events: input-only (eval mode, inputs
    requiring grad) against the full training backward (training mode, parameter gradients, inputs not requiring grad);
  * the peak allocated device memory of each.
Per-step time does not depend on the step count; 16 steps keep the run short.  The card's name and power limit are read
(read-only ``nvidia-smi`` query) in the same run.  Writes DIR/guided_completion_bench.json and prints it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

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


def timed(fn, dev):
    """(result, device ms, peak allocated MiB) of fn(), bracketed by CUDA events on the current stream."""
    torch.cuda.synchronize(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return out, e0.elapsed_time(e1), torch.cuda.max_memory_allocated(dev) / 2 ** 20


def run_batch(cfg, sd, batch, steps, repeats, w, dev):
    net = DiffuseSG(img_size=cfg["img"], in_chans=in_chans(cfg), patch_size=1, embed_dim=cfg["embed"],
                    depths=cfg["depths"], num_heads=cfg["heads"], window_size=cfg["window"], mlp_ratio=4., drop_rate=0.,
                    attn_drop_rate=0., drop_path_rate=0.0, self_condition=True, symmetric_noise=False,
                    out_chans_adj=cfg["c_e"], out_chans_node=cfg["c_n"])
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).eval()
    flags = synthetic_node_flags(cfg, batch, seed=0).to(dev)
    known = completion.encode_known(flags, cfg["c_e"], cfg["c_n"], *condition(flags.cpu(), 1), NUM_ADJ_TYPE, NUM_NODE_TYPE)
    sampler = NodeAdjEDMSampler(num_steps=steps, clip_samples=True, clip_samples_min=-1.0, clip_samples_max=1.0,
                                clip_samples_scope="x_0", dev=dev, objective="edm", self_condition=True,
                                symmetric_noise=False)
    kw = dict(num_node_chan=cfg["c_n"], num_edge_chan=cfg["c_e"])
    runs = {"unguided": lambda: sampler.sample_completion(model, flags, *known, **kw),
            "guided": lambda: sampler.sample_completion(model, flags, *known, guidance_scale=w, **kw)}
    res = {k: dict(ms_per_step=[], peak_mib=0.0) for k in runs}
    for k, fn in runs.items():          # warm-up: graph capture, TrainState, shadows
        np.random.seed(0)
        fn()
    for _ in range(repeats):
        for k, fn in runs.items():
            np.random.seed(0)
            _, ms, peak = timed(fn, dev)
            res[k]["ms_per_step"].append(ms / steps)
            res[k]["peak_mib"] = max(res[k]["peak_mib"], peak)

    # one preconditioned call's backward: input-only (eval) against the full training backward
    g = torch.Generator(device=dev).manual_seed(2)
    pair = (flags[:, None, :, None] & flags[:, None, None, :]).float()
    adj = torch.randn(batch, cfg["c_e"], cfg["img"], cfg["img"], device=dev, generator=g) * pair
    node = torch.randn(batch, cfg["img"], cfg["c_n"], device=dev, generator=g) * flags[..., None].float()
    sig = torch.full((batch,), 1.5, device=dev)
    wa, wn = torch.randn(adj.shape, device=dev, generator=g), torch.randn(node.shape, device=dev, generator=g)
    plain = NodeAdjPrecond(precond="edm", model=net, self_condition=False, symmetric_noise=False)

    def backward_ms(training):
        net.train(training)
        plain.train(training)
        a = adj.clone().requires_grad_(not training)
        x = node.clone().requires_grad_(not training)
        da, dn = plain(a, x, flags, sig, adj, node)
        loss = (da * wa).sum() + (dn * wn).sum()
        _, ms, peak = timed(loss.backward, dev)
        net.zero_grad(set_to_none=True)
        return ms, peak

    bwd = {}
    for name, training in (("input_only", False), ("training", True)):
        backward_ms(training)           # warm-up
        ms, peak = zip(*[backward_ms(training) for _ in range(repeats)])
        bwd[name] = dict(ms=list(ms), peak_mib=max(peak))
    net.eval()
    res["denoiser_backward"] = bwd
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batches", default="128,256,512,1024")
    ap.add_argument("--num-steps", type=int, default=16)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--guidance", type=float, default=0.5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("guided_completion_bench: no CUDA device (this measures the GPU; nothing to report without one)")
    dev = torch.device("cuda:0")
    cfg = CONFIGS["vg"]
    sd = synthetic_state_dict(cfg, seed=1234, stress=False)
    result = dict(workload=dict(geometry="vg", num_steps=args.num_steps, repeats=args.repeats, guidance_scale=args.guidance,
                                condition="half of the valid nodes (class + box) and the relations among them"),
                  gpu_before=gpu_info(0), batches={})
    fits = None
    for b in [int(x) for x in args.batches.split(",")]:
        try:
            result["batches"][b] = run_batch(cfg, sd, b, args.num_steps, args.repeats, args.guidance, dev)
            fits = b
        except torch.cuda.OutOfMemoryError as e:
            result["batches"][b] = dict(out_of_memory=str(e).splitlines()[0])
            break
        finally:
            torch.cuda.empty_cache()
        print(b, json.dumps(result["batches"][b]), flush=True)
    result["largest_batch_that_fits"] = fits
    result["gpu_after"] = gpu_info(0)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "guided_completion_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
