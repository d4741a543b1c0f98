#!/usr/bin/env python
"""Benchmark of the DiffuseSG sampling hot path: sampled scene graphs / second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--config vg] [--batch 512]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input: one full NodeAdjEDMSampler run (256
stochastic-Heun steps, 511 preconditioned-denoiser calls plus the data-dependent self-conditioning passes) over
`--batch` Visual-Genome-shaped graphs per GPU with seeded random-init weights (no dataset or checkpoint is
available offline).  N > 1 is launched by torchrun, one rank per GPU; the batch is sharded by sample with no
per-step communication (weak scaling: every rank samples its own `--batch` graphs).

Two numbers per step:
  value  device-resident: node flags and the initial noise are already in HBM, the result stays in HBM;
  e2e    the reference-facing call `sampler.sample(model, node_flags)` with HOST node flags: the initial noise
         is drawn on the CPU generator and uploaded (as the reference does), the samples come back as CPU tensors.

`--impl reference` times the reference's CPU implementation of the same path - the UNMODIFIED reference modules staged
under oracle/_ref by __graft_entry__.build() (oracle/stage_reference.py), all host threads - on a bounded sample of the
workload (batch 8, a few Heun steps, extrapolated by counted denoiser passes; the line's config.measured_sample says so).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from diffusesg_b200.utils.synthetic import CONFIGS, in_chans, synthetic_node_flags, synthetic_state_dict  # noqa: E402

METRIC = "sampled scene graphs/sec"
UNIT = "graphs/s"
EXPECTED_PASSES_256 = 766.5  # 511 precond calls + E[#coins < 0.5] (model/precond/precond.py:90)
GFLOP_PER_PASS = {"vg": 13.30, "coco": 7.36, "n64w16": 14.66}  # SURVEY.md 8(d): GEMM + bmm + conv, per sample


def ncu_traffic_per_launch(pattern: str):
    """Average dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernels matching `pattern`, over the
    last denoiser pass of the committed ncu launch list (profiles/, same one-pass command), or None."""
    import csv
    import re
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_launches_pass_ncu.csv")
    if not os.path.exists(path):
        return None
    rows = list(csv.reader(open(path)))
    try:
        hi = next(i for i, r in enumerate(rows) if r and r[0] == "ID")
    except StopIteration:
        return None
    hdr = rows[hi]
    col = {h: i for i, h in enumerate(hdr)}
    per = {}
    for r in rows[hi + 1:]:
        if len(r) != len(hdr):
            continue
        e = per.setdefault(int(r[col["ID"]]), {"name": r[col["Kernel Name"]], "b": 0.0})
        if r[col["Metric Name"]] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            e["b"] += float(r[col["Metric Value"]].replace(",", ""))
    ids = sorted(per)
    starts = [i for i in ids if "sinusoid_kernel" in per[i]["name"]]  # first kernel of a denoiser pass
    if not starts:
        return None
    sel = [per[i]["b"] for i in ids if i >= starts[-1] and re.search(pattern, per[i]["name"])]
    return sum(sel) / len(sel) if sel else None


def ncu_edm_traffic():
    path = os.path.join(ROOT, "profiles", "r2_ncu_edm_summary.json")
    return json.load(open(path))["dram_bytes_per_launch"] if os.path.exists(path) else None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tensor_sustained=p["bf16_tflops_sustained"], tensor_burst=p["bf16_tflops"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tensor_sustained=1400.0, tensor_burst=1590.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            try:
                pw.append(float(f[2]))
            except ValueError:
                pass
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        busy = sorted(sm)[len(sm) // 4:]  # drop idle samples at the edges
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "power_w": float(np.median(sorted(pw)[len(pw) // 4:])) if pw else None}


def build_native_model(cfg, device):
    from diffusesg_b200.model.diffusesg.diffusesg import DiffuseSG
    from diffusesg_b200.model.precond.precond import NodeAdjPrecond
    net = DiffuseSG(img_size=cfg["img"], in_chans=in_chans(cfg), patch_size=1, embed_dim=cfg["embed"],
                    depths=cfg["depths"], num_heads=[3, 6, 12, 24], window_size=cfg["window"], mlp_ratio=4.,
                    drop_rate=0., attn_drop_rate=0., drop_path_rate=0.0, self_condition=cfg["self_cond"],
                    symmetric_noise=False, out_chans_adj=cfg["c_e"], out_chans_node=cfg["c_n"])
    net.load_state_dict(synthetic_state_dict(cfg, seed=1234, stress=False), strict=True)
    return NodeAdjPrecond(precond="edm", model=net.to(device), self_condition=cfg["self_cond"],
                          symmetric_noise=False).eval()


def make_sampler(cfg, device, num_steps):
    from diffusesg_b200.runner.mcmc_sampler.edm import NodeAdjEDMSampler
    return NodeAdjEDMSampler(num_steps=num_steps, clip_samples=True, clip_samples_min=-1.0, clip_samples_max=1.0,
                             clip_samples_scope="x_0", dev=device, objective="edm", self_condition=cfg["self_cond"],
                             symmetric_noise=False)


# -----------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the staged unmodified reference on the host cores
# -----------------------------------------------------------------------------------------------------------
def cpu_reference_rate(cfg, batch, num_steps, repeats, warmup):
    """Time the reference's CPU implementation of the path on all host cores.

    Preferred: the UNMODIFIED reference staged under oracle/_ref (``NodeAdjEDMSampler.sample`` over
    ``NodeAdjPrecond(DiffuseSG)``, dev='cpu'; kind = "reference").  Only if it is not staged (a box that never saw
    /root/reference and no oracle/_ref travelled) the oracle port of the same modules runs (kind = "port").
    Returns dict(rate = graphs/s extrapolated to 256 steps by counted raw denoiser passes, ms, passes, sec_per_pass,
    kind, cores)."""
    from oracle import stage_reference as R
    torch.set_num_threads(os.cpu_count() or 1)
    sd = synthetic_state_dict(cfg, seed=1234, stress=False)
    flags = synthetic_node_flags(cfg, batch, seed=1234)
    passes = [0]
    if R.root() is not None:
        ref = R.load()
        model = R.build_network(ref, cfg, sd)
        model.model.register_forward_hook(lambda *_: passes.__setitem__(0, passes[0] + 1))
        sampler = ref.NodeAdjEDMSampler(num_steps=num_steps, clip_samples=True, clip_samples_min=-1.0,
                                        clip_samples_max=1.0, clip_samples_scope="x_0", dev="cpu", objective="edm",
                                        self_condition=cfg["self_cond"], symmetric_noise=False)
        kind = "reference"

        def run():
            sampler.sample(model=model, node_flags=flags, num_node_chan=cfg["c_n"], num_edge_chan=cfg["c_e"])
    else:
        from oracle import denoiser_oracle as O
        from oracle import edm_oracle as E
        kind = "port"

        def net(adj, node, f, labels, sa, sn):
            passes[0] += 1
            return O.denoiser_forward(sd, img=cfg["img"], embed=cfg["embed"], depths=cfg["depths"], heads=cfg["heads"],
                                      window=cfg["window"], self_condition=cfg["self_cond"], adj=adj, node=node, flags=f,
                                      noise_labels=labels, sc_adj=sa, sc_node=sn)

        pmodel = lambda a, n, f, sig, sa, sn: O.precond_forward(net, a, n, f, sig, sa, sn, coin=np.random.rand)

        def run():
            E.sample(pmodel, flags, cfg["c_e"], cfg["c_n"], num_steps=num_steps)
    times, counts = [], []
    torch.manual_seed(1234)
    np.random.seed(1234)
    with torch.no_grad():
        for it in range(warmup + repeats):
            passes[0] = 0
            t0 = time.perf_counter()
            run()
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
                counts.append(passes[0])
    sec_per_pass = sum(times) / max(1, sum(counts))
    return dict(rate=batch / (sec_per_pass * EXPECTED_PASSES_256), ms=1e3 * sum(times) / len(times),
                passes=sum(counts) / len(counts), sec_per_pass=sec_per_pass, kind=kind, cores=torch.get_num_threads())


def cpu_sample_text(args, r):
    what = ("the UNMODIFIED reference (oracle/_ref: NodeAdjEDMSampler.sample over NodeAdjPrecond(DiffuseSG), fp32, dev=cpu)"
            if r["kind"] == "reference" else "oracle port of the reference PyTorch CPU path (oracle/_ref not staged)")
    return (f"{what}, {args.config} geometry, batch {args.cpu_batch}, {args.cpu_steps} Heun steps per timed step "
            f"({r['passes']:.1f} raw denoiser passes, {r['sec_per_pass']:.3f} s/pass), extrapolated by counted passes to "
            f"256 steps = {EXPECTED_PASSES_256} expected passes per graph batch")


def run_reference(args, cfg, rank, world):
    if rank != 0:
        return
    r = cpu_reference_rate(cfg, args.cpu_batch, args.cpu_steps, args.steps, args.warmup)
    config = workload_config(args, cfg, world)
    # what this arm actually executed per timed step (the metric is extrapolated to the workload above)
    config["measured_sample"] = {"batch": args.cpu_batch, "heun_steps": args.cpu_steps, "raw_passes": r["passes"],
                                 "extrapolated_to_passes": EXPECTED_PASSES_256, "device": "cpu", "world": 1}
    line = {"impl": "reference", "metric": METRIC, "value": r["rate"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": r["rate"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                             "sample": cpu_sample_text(args, r)},
            "e2e": {"value": r["rate"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(args, cfg, world):
    return {"workload": f"DiffuseSG EDM sampling, {cfg['dataset']}-shaped synthetic graphs (N={cfg['img']}, "
                        f"C_e={cfg['c_e']}, C_n={cfg['c_n']}, window {cfg['window']}, depths {cfg['depths']}), "
                        f"{args.num_steps} stochastic Heun steps, self-conditioning coin flip on",
            "batch_per_gpu": args.batch, "global_batch": args.batch * world, "num_steps": args.num_steps,
            "parallelism": f"sample-sharded x{world}, no per-step collective",
            "l2": "working set per step (>= 6 GB of activations at batch 512) exceeds the 126 MB L2; no flush needed"}


# -----------------------------------------------------------------------------------------------------------
# native arm
# -----------------------------------------------------------------------------------------------------------
def run_native(args, cfg, rank, local_rank, world):
    from diffusesg_b200 import native
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the native path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL_DEBUG is left as the caller set it (the driver reads NCCL's INFO lines); whatever NCCL prints on
        # fd 1 lands on stderr through the fd swap in main(), so stdout still carries exactly one line
        dist.init_process_group("nccl", device_id=device)
    native.lib()
    torch.manual_seed(1234 + rank)   # the reference offsets the seed by the rank (utils/arg_parser.py:293-294)
    np.random.seed(1234 + rank)
    model = build_native_model(cfg, device)
    sampler = make_sampler(cfg, device, args.num_steps)
    B, N, ce, cn = args.batch, cfg["img"], cfg["c_e"], cfg["c_n"]
    flags_host = synthetic_node_flags(cfg, B, seed=1234 + rank)
    flags_dev = flags_host.to(device)
    elems = B * (ce * N * N + N * cn)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # device-resident step: initial noise pre-generated in HBM, result left in HBM
    init = [(torch.randn(B, ce, N, N, device=device), torch.randn(B, N, cn, device=device))
            for _ in range(2)]
    k = [0]
    last = {}

    def step_device():
        a, n = init[k[0] % 2]
        k[0] += 1
        out = sampler.sample_on_device(model, flags_dev, init_adjs=a, init_nodes=n, num_node_chan=cn, num_edge_chan=ce)
        last["adjs"], last["nodes"] = out[0], out[1]

    # e2e: the sharded entry point the reference's eval loop corresponds to (runner/sampler/sampler_node_adj.py:166-177
    # + the final gather :331-345): every rank holds the host flags of ALL world * B graphs, samples its own slice and
    # the slices are all-gathered, so at N > 1 the one collective of the path is inside the timed region
    from diffusesg_b200.runner.sampler.sharded import sample_sharded
    flags_all_host = torch.cat([synthetic_node_flags(cfg, B, seed=1234 + r) for r in range(world)])

    def step_e2e():
        a, n = sample_sharded(sampler, model, flags_all_host, world * B, cn, ce, gather_device=device)
        assert a.shape[0] == world * B and not a.is_cuda

    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()

    # end-to-end through the reference-facing API with host inputs / outputs.  Measured right after the warm-up and
    # BEFORE the device-resident steps: under the 1000 W cap the SM clock sags by ~10 % over the first two minutes of
    # sustained load (same power, rising temperature), so whichever phase runs later is slower; e2e is the headline,
    # `value` and the roofline explain it (--e2e-last restores the other order; both phases record their clocks).
    e2e_steps = max(1, min(args.steps, args.e2e_steps))

    def measure_e2e():
        step_e2e()
        p0 = model.raw_passes
        with ClockSampler(local_rank) as ck:
            ms = timed(step_e2e, e2e_steps) / e2e_steps
        return ms, (model.raw_passes - p0) / e2e_steps, ck

    if not args.e2e_last:
        ms_e2e, passes_e2e, clocks_e2e = measure_e2e()
    passes0, launches0 = model.raw_passes, native.launch_count()
    # per-kernel event brackets inside the timed region: with CUDA graphs (default) every `profile_stride`-th Heun STEP
    # is issued through the eager launch sequence (same kernels, bit-identical results) with all of its launches
    # bracketed; without graphs every `profile_stride`-th denoiser PASS is bracketed (and every EDM step launch)
    graphs = sampler.use_graphs
    if graphs:
        sampler.eager_every = args.profile_stride
    native.profile_begin(1 if graphs else args.profile_stride)
    with ClockSampler(local_rank) as clocks:
        ms_total = timed(step_device, args.steps)
    prof = native.profile_read()
    native.profile_stop()
    sampler.eager_every = 0
    passes = (model.raw_passes - passes0) / args.steps
    launches = native.launch_count() - launches0
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)

    if args.e2e_last:
        ms_e2e, passes_e2e, clocks_e2e = measure_e2e()
    e2e_value = world * B / (ms_e2e * 1e-3)

    # strong scaling beside the weak-scaling headline: the same global batch of B graphs split over the ranks
    strong = None
    if world > 1 and B % world == 0 and not args.no_strong:
        Bs = B // world
        fl_s = flags_dev[:Bs].contiguous()
        init_s = (init[0][0][:Bs].contiguous(), init[0][1][:Bs].contiguous())

        def step_strong():
            sampler.sample_on_device(model, fl_s, init_adjs=init_s[0], init_nodes=init_s[1], num_node_chan=cn,
                                     num_edge_chan=ce)
        step_strong()   # builds the plan / graphs for the smaller batch
        ms_s = timed(step_strong, 1)
        strong = {"scaling": "strong", "global_batch": B, "batch_per_gpu": Bs, "value": B / (ms_s * 1e-3), "unit": UNIT,
                  "ms_per_step": ms_s, "steps": 1, "note": "device-resident, same definition as `value`"}

    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    pk = peaks()
    g0, g1 = prof.get("gemm_tcgen05", {}), prof.get("fused_mlp_tcgen05", {})
    g = {k: g0.get(k, 0) + g1.get(k, 0) for k in ("ms", "flops", "bytes", "launches")}  # every tcgen05 launch
    # shares of the step: the denoiser classes are bracketed on every `profile_stride`-th pass only, the EDM step
    # classes on every launch -> weight the former by the stride before forming shares
    every_launch = ("edm_step", "edm_pre_step_philox")
    eff_ms = {name: c["ms"] * (1 if (graphs or name in every_launch) else args.profile_stride) for name, c in prof.items()}
    total_prof_ms = sum(eff_ms.values()) or 1.0
    gemm_tflops = g["flops"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] else 0.0
    # `roofline`: the single dominant kernel (gemm_kernel: every nn.Linear that is not inside a fused block kernel);
    # `roofline_tcgen05_class`: all tcgen05 kernels together, i.e. including the HBM-bound fused block head / tail /
    # proj + LN2 kernels whose LayerNorm / FiLM / GELU work carries no GEMM flops
    how = (f"CUDA events around every launch of every {args.profile_stride}-th Heun step (issued eagerly; all other steps are "
           "CUDA-graph replays of the same launches) inside the timed region" if graphs else
           f"CUDA events around every launch of every {args.profile_stride}-th denoiser pass inside the timed region")
    g0_tflops = g0.get("flops", 0) / (g0["ms"] * 1e-3) / 1e12 if g0.get("ms") else 0.0
    roofline = {"bound": "tensor", "kernel": "gemm_kernel<BN,EPI,PAIR> (tcgen05/TMEM/TMA; the dominant kernel of the pass)",
                "achieved": g0_tflops, "peak": pk["tensor_sustained"], "unit": "TFLOP/s", "frac": g0_tflops / pk["tensor_sustained"],
                "peak_source": pk["source"] + ", sustained bf16 (kernel timed inside a long step)",
                "traffic": ncu_traffic_per_launch(r"gemm_kernel"),
                "traffic_note": "bytes per launch, mean over the gemm_kernel launches of one denoiser pass (ncu dram__bytes_read + write, profiles/r2_launches_pass_ncu.csv)",
                "algorithmic_bytes_per_launch": g0["bytes"] / g0["launches"] if g0.get("launches") else None,
                "launches_timed": g0.get("launches"),
                "avg_launch_ms": g0["ms"] / g0["launches"] if g0.get("launches") else None,
                "share_of_profiled_time": eff_ms.get("gemm_tcgen05", 0.0) / total_prof_ms, "how": how}
    class_roof = {"bound": "tensor", "kernel": "gemm_kernel + block_head_kernel<96> + block_tail_kernel<96> + fused_mlp_kernel<192> + proj_ln_kernel<384> (every nn.Linear of the denoiser, HBM-bound K <= 192 shapes and the fused LayerNorm / FiLM / GELU work included)",
                  "achieved": gemm_tflops, "peak": pk["tensor_sustained"], "unit": "TFLOP/s", "frac": gemm_tflops / pk["tensor_sustained"],
                  "traffic": ncu_traffic_per_launch(r"gemm_kernel|block_head_kernel|block_tail_kernel|fused_mlp_kernel|proj_ln_kernel"),
                  "launches_timed": g["launches"],
                  "share_of_profiled_time": (eff_ms.get("gemm_tcgen05", 0.0) + eff_ms.get("fused_mlp_tcgen05", 0.0)) / total_prof_ms,
                  "how": how}
    classes = {}
    for name, c in prof.items():
        sec = c["ms"] * 1e-3
        classes[name] = {"launches": c["launches"], "ms": round(c["ms"], 3), "share": round(eff_ms[name] / total_prof_ms, 4),
                         "tflops": round(c["flops"] / sec / 1e12, 2) if sec and c["flops"] else None,
                         "gbs": round(c["bytes"] / sec / 1e9, 1) if sec and c["bytes"] else None}
    edm = prof.get("edm_step")
    edm_roof = None
    if edm and edm["ms"]:
        gbs = edm["bytes"] / (edm["ms"] * 1e-3) / 1e9
        edm_roof = {"bound": "hbm", "kernel": "edm_kernel<MODE> (fused Heun / Euler post step, initial mask-scale)", "achieved": gbs,
                    "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"], "traffic": ncu_edm_traffic(),
                    "traffic_note": "dram__bytes_read + write of one Heun post-step launch (ncu --set full, profiles/r2_ncu_full_edm.txt)"}
        nz = prof.get("edm_pre_step_philox")
        if nz and nz["ms"]:
            # the pre-step draws its noise in the kernel (same Philox4x32-10 / Box-Muller work as the two torch.randn_like
            # launches it replaces): ALU-bound, reported as normals per second next to its HBM rate
            edm_roof["pre_step_with_noise"] = {"kernel": "edm_pre_philox_kernel<ADJ> (x + c * eps with eps drawn in the kernel)",
                                               "bound": "alu (Philox4x32-10 + Box-Muller, bit-compatible with torch.randn_like)",
                                               "gnormals_per_s": nz["bytes"] / 8 / (nz["ms"] * 1e-3) / 1e9,
                                               "gbs": nz["bytes"] / (nz["ms"] * 1e-3) / 1e9, "launches_timed": nz["launches"]}
    flops_step = passes * GFLOP_PER_PASS.get(args.config, 0.0) * 1e9 * B
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": workload_config(args, cfg, world),
            "raw_denoiser_passes_per_step": passes, "ms_per_pass": ms_step / passes if passes else None,
            "denoiser_tflops_whole_step": flops_step / (ms_step * 1e-3) / 1e12 if flops_step else None,
            "denoiser_frac_of_sustained_peak": (flops_step / (ms_step * 1e-3) / 1e12 / pk["tensor_sustained"]) if flops_step else None,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e, "steps": e2e_steps,
                    "raw_denoiser_passes_per_step": passes_e2e, "ms_per_pass": ms_e2e / passes_e2e if passes_e2e else None,
                    "clocks": clocks_e2e.summary(),
                    # per rank: flags of all graphs + the initial noise of its slice (+ at N > 1 the slice going back up
                    # for the all-gather, as in the reference's gather_tensors); down: the slice (+ the gathered whole)
                    "h2d_bytes_per_step": int(flags_all_host.numel() + elems * 4 + (elems * 4 if world > 1 else 0)),
                    "d2h_bytes_per_step": int(elems * 4 + (world * elems * 4 if world > 1 else 0)),
                    "api": "runner.sampler.sharded.sample_sharded -> NodeAdjEDMSampler.sample per rank"
                           + (" + all_gather_into_tensor of the final samples (inside the timed region)" if world > 1 else "")},
            "gpu_launches": int(launches), "roofline": roofline, "roofline_tcgen05_class": class_roof,
            "roofline_edm_step": edm_roof, "kernel_classes": classes,
            "clocks": clocks.summary()}
    if strong is not None:
        line["strong_scaling"] = strong
    # how the launch sequence is organised (all three are on by default; each is bit-identical to its plain counterpart:
    # tests/test_gpu_denoiser.py::test_sampler_graphs_are_bit_identical, ::test_padding_skipping_matches_dense)
    plan = getattr(getattr(sampler, "_plan", None), "skip", None)
    line["schedule"] = {
        "cuda_graphs": bool(sampler.use_graphs), "fused_philox_noise": bool(sampler.fused_noise),
        "padding_skipping": None if plan is None else {
            "kept_fraction_of_compact_stage_pixels": round(plan.kept_fraction, 4),
            "level2_kept_fraction": round(plan.level2[4], 4) if plan.level2 else None,
            "note": "un-shifted stages run only on each sample's corner that can hold valid nodes (DESIGN.md 3.3); outputs "
                    "identical to the dense schedule; `roofline` counts the flops actually executed, "
                    "`denoiser_tflops_whole_step` the reference's dense flops (an effective rate)"}}
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_rate(cfg, args.cpu_batch, args.cpu_steps, 1, 0)
        line["cpu_baseline"] = {"value": r["rate"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                                "sample": cpu_sample_text(args, r)}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 63 * 10**6   # sample data; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Write the samples of the last timed step (what ``sample_on_device`` returned) as float32 ``<name>.npy``.
    Over DUMP_LIMIT_BYTES in all, the same seeded subset of graphs is kept from every array."""
    b = next(iter(outputs.values())).shape[0]
    per_graph = sum(t[0].numel() * 4 for t in outputs.values())
    keep = min(b, DUMP_LIMIT_BYTES // per_graph)
    idx = torch.arange(b) if keep == b else torch.from_numpy(np.sort(np.random.default_rng(0).choice(b, keep, replace=False)))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t[idx.to(t.device)].float().cpu().numpy())
    print(f"bench.py: wrote {', '.join(outputs)} of {keep} of {b} graphs to {out_dir}", file=sys.stderr)


_RESULT_FD = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    # Everything else that lands on fd 1 (NCCL's version banner is printed from C at every debug level but NONE,
    # library chatter) goes to stderr, so that stdout carries exactly one line.
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="vg", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=512, help="graphs per GPU per step")
    ap.add_argument("--num-steps", type=int, default=256, help="EDM sampler steps (mcmc.num_steps)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--profile-stride", type=int, default=16)
    ap.add_argument("--cpu-batch", type=int, default=8)
    ap.add_argument("--cpu-steps", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-last", action="store_true", help="measure e2e after the device-resident steps (default: before)")
    ap.add_argument("--no-strong", action="store_true", help="skip the extra strong-scaling step at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the final samples of the last timed step (rank 0) as DIR/adjs.npy, DIR/nodes.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the native path's samples; use it with --impl native")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
    else:
        run_native(args, cfg, rank, local_rank, world)


if __name__ == "__main__":
    main()
