"""Drop-in ``NodeAdjEDMSampler``: the 256-step stochastic Heun loop on fused native kernels.

Interface of runner/mcmc_sampler/edm.py:231-445 of the reference: keyword-only constructor with the same names
and defaults, ``sample(model, node_flags, init_adjs=None, init_nodes=None, sanity_check_gt_adjs=None, ...)`` with
the same return convention ((adjs, nodes) on the CPU, or the 4-tuple with interim snapshots), the same consumption
order of the global torch RNGs (CPU generator for the initial sample, device generator per step, adjacency
before nodes) and of the numpy RNG (through the model's coin flip).

What changed underneath:
* the sigma grid and every per-step scalar (gamma, t_hat, noise coefficient, h, 1/t) are evaluated once on the
  host with the reference's own fp32/fp64 tensor expressions - no 0-d device tensors, no per-step host sync
  (the reference syncs twice per step: edm.py:355 and :433);
* each step is two fused elementwise launches (libdsg_b200: dsg_edm_pre_step / dsg_edm_post_step) around the
  denoiser calls instead of ~113 ATen launches; masking is part of those kernels;
* interim snapshots are copied to pinned host memory asynchronously;
* by default every step is ONE CUDA-graph launch (graphs.py: six graphs cover the coin-flip variants of a step;
  bit-identical to the eager launch sequence; ``DSG_NO_GRAPH=1`` or any noise-replay hook keeps the eager path);
* ``sample_decoded`` fuses the reference's post-sampling decode (runner/sampler/sampler_node_adj.py:199-285) into the
  last step, so only int32 classes and four box floats per node leave the GPU (SURVEY 8f-1).

Beyond the reference: ``sample_completion`` samples with a set of state entries held at known clean values
(scene-graph completion; completion.py builds the conditions, DESIGN.md §3.6), optionally with reconstruction
guidance (``guidance_scale > 0``, DESIGN.md §3.7).
"""
from __future__ import annotations

import contextlib
import functools
import logging
import math
import os
from typing import List, Optional

import numpy as np
import torch
import torch.nn as nn

from ... import native

_TORCH_RANDN_LIKE = torch.randn_like
_TORCH_RANDN = torch.randn
from .graphs import HeunGraphPlan
from ..objectives.edm import get_edm_params, get_edm_sigma_deriv_t, get_edm_sigma_from_t, get_edm_t_from_sigma


class NodeAdjEDMSampler:
    def __init__(self, *, sigma_min=None, sigma_max=None, solver="heun", discretization="edm", schedule="linear",
                 scaling="none", C_1=0.001, C_2=0.008, M=1000, alpha=1, num_steps=256, S_churn=40, S_min=0.05,
                 S_max=50, S_noise=1.003, clip_samples, clip_samples_min, clip_samples_max, clip_samples_scope,
                 self_condition, dev, objective="edm", symmetric_noise=True):
        if (solver, discretization, schedule, scaling) != ("heun", "edm", "linear", "none") or alpha != 1:
            raise NotImplementedError("NodeAdjEDMSampler (B200): only solver='heun', discretization='edm', "
                                      "schedule='linear', scaling='none', alpha=1 (the reference defaults, "
                                      "edm.py:239-245) are built")
        if objective != "edm":
            raise NotImplementedError("objective must be 'edm'")
        if symmetric_noise:
            raise NotImplementedError("symmetric_noise=True: get_mc_sampler always passes False "
                                      "(utils/sampling_utils.py:23)")
        if clip_samples:
            assert clip_samples_scope == "x_0"  # parsed and asserted, never applied by the reference (edm.py:30)
        self.objective = objective
        self.clip_samples, self.clip_samples_min, self.clip_samples_max = clip_samples, clip_samples_min, clip_samples_max
        self.clip_samples_scope = clip_samples_scope
        self.self_condition = self_condition
        self.symmetric_noise = symmetric_noise
        self.dev = torch.device(dev) if not isinstance(dev, torch.device) else dev
        self.edm_params = get_edm_params()
        self.num_steps, self.S_churn, self.S_min, self.S_max, self.S_noise = num_steps, S_churn, S_min, S_max, S_noise
        self.solver, self.alpha = solver, alpha
        sigma_min = self.edm_params.sigma_min_sampling if sigma_min is None else sigma_min
        sigma_max = self.edm_params.sigma_max_sampling if sigma_max is None else sigma_max
        self.sigma_min, self.sigma_max = sigma_min, sigma_max
        # Karras grid in fp64 (edm.py:70, :84-88); kept on the host
        rho = self.edm_params.rho
        step_indices = torch.arange(num_steps, dtype=torch.float64)
        self.sigma_steps = (sigma_max ** (1 / rho) + step_indices / (num_steps - 1) *
                            (sigma_min ** (1 / rho) - sigma_max ** (1 / rho))) ** rho
        self.sigma, self.sigma_deriv, self.sigma_inv = get_edm_sigma_from_t, get_edm_sigma_deriv_t, get_edm_t_from_sigma
        self.s = lambda t: 1
        self.s_deriv = lambda t: 0
        self.last_raw_passes = 0
        # Draw the per-step noise inside the fused pre-step kernel (bit-identical to the reference's randn_like calls
        # and generator advance; SURVEY 8f-3).  DSG_NO_FUSED_NOISE=1 keeps the two torch.randn_like launches.
        self.fused_noise = os.environ.get("DSG_NO_FUSED_NOISE", "0") != "1"
        # One CUDA-graph launch per step (graphs.py).  `eager_every = k > 0` runs every k-th step through the eager
        # launch sequence instead (same kernels, same results) so that per-kernel event brackets can be taken inside
        # a timed region (bench.py).
        self.use_graphs = os.environ.get("DSG_NO_GRAPH", "0") != "1"
        self.eager_every = 0
        self._plan = None
        # Padded-row skipping (SURVEY 8f-4, include/dsg_b200.h: dsg_model_skip_info): the un-shifted leading stages of
        # the denoiser run only on the image rows that can hold valid nodes.  DSG_NO_SKIP=1 keeps the dense schedule.
        self.skip_padding = os.environ.get("DSG_NO_SKIP", "0") != "1"

    # ------------------------------------------------------------------------------------------------------
    def step_scalars(self, t_cur: torch.Tensor, t_next: torch.Tensor) -> dict:
        """Every scalar one loop iteration derives from (t_cur, t_next), with the reference's expressions on
        0-d CPU tensors (edm.py:355-356, :361, :369, :384-391, :414), returned as python floats."""
        gamma = min(self.S_churn / self.num_steps, np.sqrt(2) - 1) if self.S_min <= self.sigma(t_cur) <= self.S_max else 0
        t_hat = self.sigma_inv(torch.as_tensor(self.sigma(t_cur) + gamma * self.sigma(t_cur)))
        noise_coef = (self.sigma(t_hat) ** 2 - self.sigma(t_cur) ** 2).clip(min=0).sqrt() * self.s(t_hat) * self.S_noise
        h = t_next - t_hat
        inv_t_hat = self.sigma_deriv(t_hat) / self.sigma(t_hat) + self.s_deriv(t_hat) / self.s(t_hat)
        t_prime = t_hat + self.alpha * h
        inv_t_prime = (self.sigma_deriv(t_prime) / self.sigma(t_prime)) if float(t_prime) != 0.0 else torch.zeros(())
        return dict(gamma=float(gamma), t_hat=t_hat, noise_coef=float(noise_coef), h=float(h),
                    inv_t_hat=float(inv_t_hat), inv_t_prime=float(inv_t_prime))

    def gen_init_sample(self, node_flags, folded_norm=False, flag_node_multi_channel=False,
                        flag_adj_multi_channel=False, num_node_chan=150, num_edge_chan=51):
        """Unit-variance start drawn on the CPU generator, adjacency first (edm.py:257-289), masked on device."""
        batch_size, max_node_num = node_flags.shape[:2]
        # torch.randn(size) IS torch.empty(size).normal_() on the default CPU generator (same stream, same values); the
        # draws go straight into pinned staging buffers that are reused from call to call (no page faults, async H2D)
        if torch.randn is not _TORCH_RANDN:   # a patched torch.randn (noise recording / replay hooks) is honoured
            init_adjs = torch.randn((batch_size, num_edge_chan, max_node_num, max_node_num)).to(self.dev, non_blocking=True)
            init_nodes = torch.randn((batch_size, max_node_num, num_node_chan)).to(self.dev, non_blocking=True)
            flags = node_flags.to(self.dev).to(torch.bool).contiguous()
            return native.edm_mask_scale(init_adjs, init_nodes, flags, 1.0)
        host_a = self._staging("init_a", (batch_size, num_edge_chan, max_node_num, max_node_num))
        host_n = self._staging("init_n", (batch_size, max_node_num, num_node_chan))
        if self.dev.type == "cuda":
            torch.cuda.current_stream(self.dev).synchronize()   # the previous call's upload has left the buffers
        init_adjs = host_a.normal_().to(self.dev, non_blocking=True)
        init_nodes = host_n.normal_().to(self.dev, non_blocking=True)
        flags = node_flags.to(self.dev).to(torch.bool).contiguous()   # any flag dtype, like mask_adjs' logical_not
        return native.edm_mask_scale(init_adjs, init_nodes, flags, 1.0)

    def _staging(self, name, shape):
        cache = self.__dict__.setdefault("_staging_bufs", {})
        buf = cache.get(name)
        if buf is None or tuple(buf.shape) != tuple(shape):
            buf = torch.empty(shape, dtype=torch.float32, pin_memory=self.dev.type == "cuda")
            cache[name] = buf
        return buf

    @staticmethod
    def _to_host(*tensors):
        """Device -> freshly allocated pinned host tensors (torch's caching host allocator recycles the blocks), one
        synchronisation for all of them."""
        outs = []
        for t in tensors:
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            h.copy_(t, non_blocking=True)
            outs.append(h)
        torch.cuda.current_stream(tensors[0].device).synchronize()
        return outs

    @torch.no_grad()
    def sample(self, model, node_flags, init_adjs=None, init_nodes=None, sanity_check_gt_adjs=None,
               sanity_check_gt_nodes=None, flag_interim_adjs=False, max_num_interim_adjs=None, flag_use_double=False,
               flag_node_multi_channel=False, flag_adj_multi_channel=False, num_node_chan=150, num_edge_chan=51):
        """Reference entry point (edm.py:291-445): returns CPU tensors."""
        out = self.sample_on_device(model, node_flags, init_adjs, init_nodes, sanity_check_gt_adjs,
                                    sanity_check_gt_nodes, flag_interim_adjs, max_num_interim_adjs, flag_use_double,
                                    flag_adj_multi_channel, num_node_chan, num_edge_chan)
        adjs, nodes, snaps_a, snaps_n = out
        adjs_cpu, nodes_cpu = self._to_host(adjs, nodes)  # synchronises the stream: the pinned snapshots are complete too
        if flag_interim_adjs:
            if flag_adj_multi_channel:
                return adjs_cpu, nodes_cpu, [None], torch.stack(snaps_n)
            return adjs_cpu, nodes_cpu, torch.stack(snaps_a), torch.stack(snaps_n)
        return adjs_cpu, nodes_cpu

    @torch.no_grad()
    def sample_decoded(self, model, node_flags, num_adj_type, num_node_type, init_adjs=None, init_nodes=None,
                       num_node_chan=150, num_edge_chan=51, return_state=False):
        """``sample`` followed by the reference's decode of the final sample for the 'bits' encodings
        (runner/sampler/sampler_node_adj.py:199-285: clamp -> sign -> bin2dec (MSB first) -> clamp to the class
        range, self-loops removed, boxes * 0.5 + 0.5, all masked), with the decode fused into the last Euler step.

        ``num_adj_type`` / ``num_node_type`` are the reference's ``raw_num_adj_type`` / ``raw_num_node_type``
        (utils/sg_utils.py:348-409).  Returns CPU tensors ``(q_adj int32 [B,N,N], q_node int32 [B,N], bbox fp32
        [B,N,4])``, preceded by the raw fp32 ``(adjs, nodes)`` when ``return_state``.  Consumes the RNG streams
        exactly like ``sample``."""
        out = self.sample_on_device(model, node_flags, init_adjs, init_nodes, num_node_chan=num_node_chan,
                                    num_edge_chan=num_edge_chan,
                                    decode=(int(num_adj_type), int(num_node_type), bool(return_state)))
        adjs, nodes, _, _, (q_adj, q_node, bbox) = out
        if return_state:
            return tuple(self._to_host(adjs, nodes, q_adj, q_node, bbox))
        return tuple(self._to_host(q_adj, q_node, bbox))

    @torch.no_grad()
    def sample_completion(self, model, node_flags, known_adj, known_node, init_adjs=None, init_nodes=None,
                          num_node_chan=150, num_edge_chan=51, decode=None, guidance_scale=0.0):
        """``sample`` with the finite entries of ``known_adj [B, C_e, N, N]`` / ``known_node [B, N, C_n]`` (fp32, NaN =
        free entry; completion.encode_known builds them from classes and boxes) held at those clean values:

        * every pre-step replaces a known entry by ``k + t_hat * eps`` (replacement at the step's noise level, with the
          eps the free entries get), a free one gets the usual ``x + noise_coef * eps``;
        * after the last step the known entries are set to ``k``: the final state carries them exactly.

        The denoiser, the Heun updates and self-conditioning are unchanged, and the RNG streams are consumed exactly as
        by ``sample`` (all-NaN ``known`` reproduces ``sample`` bit for bit).  The state between steps - what interim
        snapshots would show - is the state after each post-step, so known entries there are noisy, not ``k``.
        A finite known value outside a valid node / pair (``node_flags``) is a ValueError.

        ``guidance_scale = w > 0`` adds reconstruction guidance (Ho et al. 2022, Video Diffusion Models §3.1; DESIGN.md
        §3.7): both denoiser calls of a step (D1 and D2, at x_hat) return ``D~ = mask(D - w grad_x_hat 1/2 sum_known
        (D(x_hat) - k)^2)``, which replaces D in the Heun update and the self-conditioning hand-off.  The gradient runs
        through the native denoiser backward (the model must be the native ``NodeAdjPrecond`` / ``DiffuseSG``, in eval
        mode as for sampling); the self-conditioning inputs and the coin-flip refresh pass are constants for it.  The
        guided loop is eager and dense (no CUDA graphs, no padding skipping) and consumes the RNG streams as the unguided
        one.  ``w = 0`` is the unguided path, unchanged; a negative or non-finite ``w`` is a ValueError.

        Returns CPU ``(adjs, nodes)``, or with ``decode=(num_adj_type, num_node_type)`` the ``(q_adj, q_node, bbox)`` of
        ``sample_decoded``."""
        w = float(guidance_scale)
        if not math.isfinite(w) or w < 0.0:
            raise ValueError(f"guidance_scale must be finite and >= 0, got {guidance_scale!r}")
        known = self._check_known(node_flags, known_adj, known_node, num_edge_chan, num_node_chan)
        dec = None if decode is None else (int(decode[0]), int(decode[1]), False)
        out = self._sample_on_device(model, node_flags, init_adjs, init_nodes, num_node_chan=num_node_chan,
                                     num_edge_chan=num_edge_chan, decode=dec, known=known, guidance=w)
        if decode is None:
            return tuple(self._to_host(out[0], out[1]))
        return tuple(self._to_host(*out[4]))

    def _check_known(self, node_flags, known_adj, known_node, num_edge_chan, num_node_chan):
        """Validate a NaN-coded condition (before any kernel runs) and move it to the sampler's device."""
        if node_flags.dim() != 2:
            raise ValueError(f"node_flags: shape {tuple(node_flags.shape)}, expected [B, N]")
        b, n = node_flags.shape
        for name, t, shape in (("known_adj", known_adj, (b, num_edge_chan, n, n)), ("known_node", known_node,
                                                                                     (b, n, num_node_chan))):
            if tuple(t.shape) != shape:
                raise ValueError(f"{name}: shape {tuple(t.shape)}, expected {shape}")
            if not t.dtype.is_floating_point:
                raise ValueError(f"{name}: floating-point values expected (NaN = free), got {t.dtype}")
            if bool(t.isinf().any()):
                raise ValueError(f"{name}: infinite value (known entries are finite, free ones NaN)")
        flags = node_flags.to(known_adj.device).bool()
        pair = flags[:, None, :, None] & flags[:, None, None, :]
        if bool((~known_adj.isnan() & ~pair).any()):
            raise ValueError("known_adj: a known value on a pair with a node whose flag is 0")
        if bool((~known_node.isnan() & ~flags.to(known_node.device)[:, :, None]).any()):
            raise ValueError("known_node: a known value on a node whose flag is 0")
        return (native.require_cuda(known_adj.to(self.dev), "known_adj"),
                native.require_cuda(known_node.to(self.dev), "known_node"))

    @staticmethod
    def _unwrap(model):
        if isinstance(model, (nn.DataParallel, nn.parallel.DistributedDataParallel)):
            return model.module
        return model

    def _graph_plan(self, model, batch, n, c_e, c_n):
        """The CUDA-graph plan for (model, shapes), or None when the model is not the native preconditioner."""
        from ...model.diffusesg.diffusesg import DiffuseSG
        from ...model.precond.precond import NodeAdjPrecond
        pre = self._unwrap(model)
        if not isinstance(pre, NodeAdjPrecond) or not isinstance(pre.model, DiffuseSG):
            return None, None
        nat = pre.model._native(self.dev)
        key = (id(nat), batch, n, c_e, c_n, self.num_steps, bool(pre.self_condition))
        if self._plan is None or self._plan.key != key:
            self._plan = None   # release the old plan's buffers first
            self._plan = HeunGraphPlan(pre.model, nat, batch, n, c_e, c_n, self.num_steps, pre.self_condition, self.dev)
        return self._plan, pre

    @torch.no_grad()
    def sample_on_device(self, model, node_flags, init_adjs=None, init_nodes=None, sanity_check_gt_adjs=None,
                         sanity_check_gt_nodes=None, flag_interim_adjs=False, max_num_interim_adjs=None,
                         flag_use_double=False, flag_adj_multi_channel=False, num_node_chan=150, num_edge_chan=51,
                         decode=None):
        """The sampling loop proper; the final state stays on the device (no host sync anywhere inside).
        Returns (adjs, nodes, pinned adjacency snapshots, pinned node snapshots) - plus, with
        ``decode=(num_adj_type, num_node_type, want_state)``, the tuple (adj classes, node classes, boxes) of the
        fused last step (adjs / nodes are None unless want_state)."""
        return self._sample_on_device(model, node_flags, init_adjs, init_nodes, sanity_check_gt_adjs,
                                      sanity_check_gt_nodes, flag_interim_adjs, max_num_interim_adjs, flag_use_double,
                                      flag_adj_multi_channel, num_node_chan, num_edge_chan, decode)

    def _sample_on_device(self, model, node_flags, init_adjs=None, init_nodes=None, sanity_check_gt_adjs=None,
                          sanity_check_gt_nodes=None, flag_interim_adjs=False, max_num_interim_adjs=None,
                          flag_use_double=False, flag_adj_multi_channel=False, num_node_chan=150, num_edge_chan=51,
                          decode=None, known=None, guidance=0.0):
        """sample_on_device, with ``known = (known_adj, known_node)`` on the device for completion (the state of
        the last step is then always written; decoded outputs come from it) and ``guidance`` its reconstruction-guidance
        scale (> 0: the eager, dense loop)."""
        if known is not None and sanity_check_gt_adjs is not None:
            raise ValueError("sanity_check_gt_* (the known-answer mode) cannot be combined with known entries")
        if flag_use_double:
            raise NotImplementedError("flag_use_double: the native state is fp32 (the reference default)")
        func_round_sigma = self._unwrap(model).round_sigma
        t_steps = self.sigma_inv(func_round_sigma(self.sigma_steps))
        t_steps = torch.cat([t_steps, torch.zeros_like(t_steps[:1])]).to(torch.float32)  # t_N = 0 (edm.py:318-323)

        dev = self.dev
        flags = node_flags.to(dev).to(torch.bool).contiguous()
        if init_adjs is None or init_nodes is None:
            init_adjs, init_nodes = self.gen_init_sample(node_flags, num_node_chan=num_node_chan,
                                                         num_edge_chan=num_edge_chan)
        adjs = native.require_cuda(init_adjs.to(dev), "init_adjs")
        nodes = native.require_cuda(init_nodes.to(dev), "init_nodes")
        if adjs.dim() != 4 or nodes.dim() != 3:
            raise NotImplementedError("single-channel ([B,N,N] / [B,N]) states are not part of the scene-graph path")
        snaps_a: List[torch.Tensor] = [self._snapshot(adjs)] if flag_interim_adjs and not flag_adj_multi_channel else []
        snaps_n: List[torch.Tensor] = [self._snapshot(nodes)] if flag_interim_adjs else []
        if max_num_interim_adjs is None:
            timesteps_snapshot = set(np.arange(self.num_steps).tolist())
        else:
            timesteps_snapshot = set(np.linspace(0, self.num_steps, max_num_interim_adjs).astype(int)
                                     .clip(max=self.num_steps - 1).tolist())
        gt = None
        if sanity_check_gt_adjs is not None:
            gt = native.edm_mask_scale(native.require_cuda(sanity_check_gt_adjs.to(dev), "sanity_check_gt_adjs"),
                                       native.require_cuda(sanity_check_gt_nodes.to(dev), "sanity_check_gt_nodes"),
                                       flags, 1.0)
        passes0 = getattr(self._unwrap(model), "raw_passes", 0)

        # x_0 = init * sigma(t_0) s(t_0)                                     (edm.py:343-347)
        adjs, nodes = native.edm_mask_scale(adjs, nodes, flags, float(self.sigma(t_steps[0]) * self.s(t_steps[0])))
        # all per-step scalars up front (host), the noise levels uploaded once: no per-step H2D copy or sync
        scalars = [self.step_scalars(t_steps[i], t_steps[i + 1]) for i in range(self.num_steps)]
        # a patched randn_like (noise replay) wins; so does a torch whose normal_ launch policy moved (self-check)
        fused = self.fused_noise and torch.randn_like is _TORCH_RANDN_LIKE and native.fused_noise_ok(dev)
        net = getattr(self._unwrap(model), "model", None)
        frozen = net.frozen_weights() if hasattr(net, "frozen_weights") else contextlib.nullcontext()
        with frozen:   # the weights cannot change inside the loop: staleness is probed once, on the first call
            plan = pre = None
            if self.use_graphs and fused and gt is None and guidance == 0.0:
                plan, pre = self._graph_plan(model, adjs.shape[0], adjs.shape[2], adjs.shape[1], nodes.shape[2])
            if plan is not None:
                plan.set_flags(flags, self.skip_padding)
                out = self._loop_graphs(plan, pre, adjs, nodes, flags, scalars, flag_interim_adjs,
                                        flag_adj_multi_channel, timesteps_snapshot, snaps_a, snaps_n, decode, known)
            else:
                skip = None
                if self.skip_padding and gt is None and guidance == 0.0 and hasattr(net, "make_skip_plan"):
                    skip = net.make_skip_plan(flags, dev)
                with (net.skipping(skip) if skip is not None else contextlib.nullcontext()):
                    out = self._loop_eager(model, adjs, nodes, flags, scalars, gt, fused, flag_interim_adjs,
                                           flag_adj_multi_channel, timesteps_snapshot, snaps_a, snaps_n, decode, known,
                                           guidance)
        self.last_raw_passes = getattr(self._unwrap(model), "raw_passes", 0) - passes0
        logging.info("Done with EDM-NodeAdj MCMC.")
        return out

    def _loop_eager(self, model, adjs, nodes, flags, scalars, gt, fused, flag_interim_adjs, flag_adj_multi_channel,
                    timesteps_snapshot, snaps_a, snaps_n, decode, known=None, guidance=0.0):
        dev = self.dev
        sc_a = sc_n = None
        if guidance > 0.0:
            model = functools.partial(self._guided_call, model, known, guidance)
        t_hat_dev = torch.stack([s["t_hat"] for s in scalars]).to(torch.float32).to(dev)
        decoded = None
        for i in range(self.num_steps):
            sc = scalars[i]
            # temporary noise increase; adjacency noise is drawn first        (edm.py:355-366)
            if fused:
                # the two randn_like draws happen inside the kernel, from (and advancing) the same generator state
                if known is None:
                    adjs_hat, nodes_hat = native.edm_pre_step_fused_noise(adjs, nodes, flags, sc["noise_coef"])
                else:
                    adjs_hat, nodes_hat = native.edm_pre_step_fused_noise_known(adjs, nodes, known, flags,
                                                                                sc["noise_coef"], float(sc["t_hat"]))
            else:
                eps_a = torch.randn_like(adjs)
                eps_n = torch.randn_like(nodes)
                if known is None:
                    adjs_hat, nodes_hat = native.edm_pre_step(adjs, nodes, eps_a, eps_n, flags, sc["noise_coef"])
                else:
                    adjs_hat, nodes_hat = native.edm_pre_step_known(adjs, nodes, eps_a, eps_n, known, flags,
                                                                    sc["noise_coef"], float(sc["t_hat"]))
            sigma_tensors = t_hat_dev[i].view(-1).expand(flags.size(0))
            d1 = gt if gt is not None else model(adjs_hat, nodes_hat, flags, sigma_tensors, sc_a, sc_n)
            if i == self.num_steps - 1:
                if decode is None or known is not None:
                    adjs, nodes = native.edm_post_step(adjs_hat, nodes_hat, d1, None, flags, sc["inv_t_hat"], sc["h"], 0.0)
                    if known is not None:
                        native.edm_apply_known(adjs, nodes, known, flags)
                        if decode is not None:
                            decoded = native.decode_samples(adjs, nodes, flags, decode[0], decode[1])
                else:
                    adjs, nodes, *decoded = native.edm_final_step_decode(adjs_hat, nodes_hat, d1, flags, sc["inv_t_hat"],
                                                                         sc["h"], decode[0], decode[1], decode[2])
                d2 = d1
            else:
                # second evaluation at (x_hat, t_hat) again, self-conditioned on D1 (edm.py:400-405)
                if gt is None:
                    if self.self_condition:
                        sc_a, sc_n = d1
                    else:
                        sc_a = sc_n = None
                    d2 = model(adjs_hat, nodes_hat, flags, sigma_tensors, sc_a, sc_n)
                else:
                    d2 = gt
                adjs, nodes = native.edm_post_step(adjs_hat, nodes_hat, d1, d2, flags, sc["inv_t_hat"], sc["h"],
                                                   sc["inv_t_prime"])
            sc_a, sc_n = d2 if self.self_condition else (None, None)
            if flag_interim_adjs and i in timesteps_snapshot and adjs is not None:
                if not flag_adj_multi_channel:
                    snaps_a.append(self._snapshot(adjs))
                snaps_n.append(self._snapshot(nodes))
        if decode is not None:
            return adjs, nodes, snaps_a, snaps_n, tuple(decoded)
        return adjs, nodes, snaps_a, snaps_n

    @staticmethod
    def _guided_call(model, known, w, adjs_hat, nodes_hat, flags, sigmas, sc_a, sc_n):
        """D~ = mask(D - w G), G = grad_x_hat 1/2 sum_known (D(x_hat) - k)^2: the denoiser's backward with the residual
        mask(isnan(k) ? 0 : D - k) as its output gradient (native kernels for both elementwise steps)."""
        xa = adjs_hat.detach().requires_grad_(True)
        xn = nodes_hat.detach().requires_grad_(True)
        with torch.enable_grad():
            da, dn = model(xa, xn, flags, sigmas, sc_a, sc_n)
            ra, rn = native.edm_guidance_residual(da.detach(), dn.detach(), known, flags)
            ga, gn = torch.autograd.grad((da, dn), (xa, xn), (ra, rn))
        return native.edm_guidance_update(da.detach(), dn.detach(), ga, gn, flags, w)

    def _loop_graphs(self, plan, pre, adjs, nodes, flags, scalars, flag_interim_adjs, flag_adj_multi_channel,
                     timesteps_snapshot, snaps_a, snaps_n, decode, known=None):
        """One graph launch per step; the coins are drawn here, in the order NodeAdjPrecond.forward would draw them
        (model/precond/precond.py:90: one per preconditioned call, only when the model self-conditions)."""
        dev = self.dev
        gen = torch.cuda.default_generators[dev.index if dev.index is not None else torch.cuda.current_device()]
        seed, off0 = gen.initial_seed(), gen.get_offset()
        plan.X[0].copy_(adjs)
        plan.X[1].copy_(nodes)
        plan.set_known(known)
        if plan.self_condition:
            plan.SC[0].zero_()   # "no self-conditioning yet" is a zero tensor (diffusesg.py:786-789)
            plan.SC[1].zero_()
        off_end = plan.begin(scalars, seed, off0)
        coin = (lambda: np.random.rand() < 0.5) if pre.self_condition else (lambda: False)
        last_i = self.num_steps - 1
        for i in range(self.num_steps):
            last = i == last_i
            c1 = coin()
            c2 = False if last else coin()
            if self.eager_every and i % self.eager_every == self.eager_every - 1 and not (last and decode is not None):
                pre.raw_passes += self._eager_step_on_plan(plan, pre, scalars[i], c1, c2, last,
                                                           plan.step_offset(off0, i), gen, known is not None)
            else:
                pre.raw_passes += plan.replay(c1, c2, last, decode if last else None, known is not None)
            if flag_interim_adjs and i in timesteps_snapshot and not (last and decode is not None and not decode[2]):
                if not flag_adj_multi_channel:
                    snaps_a.append(self._snapshot(plan.X[0]))
                snaps_n.append(self._snapshot(plan.X[1]))
        gen.set_offset(off_end)
        if decode is not None:
            state = (plan.X[0].clone(), plan.X[1].clone()) if decode[2] else (None, None)
            return state + (snaps_a, snaps_n, (plan.adj_cls.clone(), plan.node_cls.clone(), plan.bbox.clone()))
        return plan.X[0].clone(), plan.X[1].clone(), snaps_a, snaps_n

    def _eager_step_on_plan(self, plan, pre, sc, c1, c2, last, offset, gen, known=False):
        """The launches of one step issued eagerly on the plan's buffers (profiling: per-kernel event brackets);
        ``known``: completion with the condition in plan.K."""
        net, nat = plan.net, plan.nat
        plan.advance_only()
        gen.set_offset(offset)
        if known:
            xh = native.edm_pre_step_fused_noise_known(plan.X[0], plan.X[1], plan.K, plan.flags, sc["noise_coef"],
                                                       float(sc["t_hat"]))
        else:
            xh = native.edm_pre_step_fused_noise(plan.X[0], plan.X[1], plan.flags, sc["noise_coef"])
        plan.XH[0].copy_(xh[0])
        plan.XH[1].copy_(xh[1])
        scp = plan.SC if plan.self_condition else (None, None)

        def D(scin, out):
            net.denoise_into(nat, plan.XH[0], plan.XH[1], plan.flags, plan.sigma, scin[0], scin[1], out[0], out[1],
                             plan.skip)

        if c1:
            D(scp, plan.T)
            D(plan.T, plan.D1)
        else:
            D(scp, plan.D1)
        if last:
            x = native.edm_post_step(plan.XH[0], plan.XH[1], plan.D1, None, plan.flags, sc["inv_t_hat"], sc["h"], 0.0)
            n = 1 + int(c1)
        else:
            sc2 = plan.D1 if plan.self_condition else (None, None)
            if c2:
                D(sc2, plan.T)
                D(plan.T, plan.SC)
            else:
                D(sc2, plan.SC)
            x = native.edm_post_step(plan.XH[0], plan.XH[1], plan.D1, plan.SC, plan.flags, sc["inv_t_hat"], sc["h"],
                                     sc["inv_t_prime"])
            n = 2 + int(c1) + int(c2)
        plan.X[0].copy_(x[0])
        plan.X[1].copy_(x[1])
        if known and last:
            native.edm_apply_known(plan.X[0], plan.X[1], plan.K, plan.flags)
        return n

    @staticmethod
    def _snapshot(t: torch.Tensor) -> torch.Tensor:
        host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        host.copy_(t, non_blocking=True)
        return host

    @staticmethod
    def get_num_edges(adjs, node_flags, threshold=0.0):
        """runner/mcmc_sampler/__init__.py:50 (diagnostic only; no longer called inside the loop)."""
        valid = node_flags[:, None, :, None] & node_flags[:, None, None, :]
        return ((adjs > threshold) & valid).flatten(1).sum(-1).float()
