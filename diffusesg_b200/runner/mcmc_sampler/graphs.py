"""CUDA-graph replay of the stochastic-Heun loop (one graph launch per sampler step).

One reference step (runner/mcmc_sampler/edm.py:350-434) is: noise injection, 1-2 preconditioned denoiser calls - each
preceded, with probability 1/2, by the self-conditioning refresh pass of model/precond/precond.py:90-98 - and the
Heun / Euler update: 190-380 kernel launches issued from Python through ctypes.  The launch sequence depends only on
the two coin flips of the step (drawn on the host from the numpy stream, in the reference's order) and on whether it
is the last step, so six graphs cover every step.  Per-step scalars (noise coefficient, 1/t_hat, h, 1/t', t_hat and
the Philox counter offsets of the step's two ``randn_like`` draws) cannot be baked into a captured launch: they live
in a device table, one ``dsg_edm_step_params`` row per step, and the first node of every graph copies the current row
into the struct all other nodes read (``dsg_edm_step_advance``).

Fixed buffers (pointers are part of the captured launches):
    X   state            XH  x_hat            D1  first denoiser output
    SC  self-conditioning carried between steps == the step's last denoiser output (D2 is written into it)
    T   output of a coin-flip refresh pass
Step (c1, c2 = the two coins):
    XH = mask(X + c * eps)
    c1:  T  = D(XH; SC);  D1 = D(XH; T)        else  D1 = D(XH; SC)
    c2:  T  = D(XH; D1);  SC = D(XH; T)        else  SC = D(XH; D1)        (not on the last step)
    X  = heun(XH, D1, SC)                            X = euler(XH, D1) [+ decode] on the last step
The kernels, their order and their arithmetic are those of the eager path: results are bit-identical
(tests/test_gpu_denoiser.py::test_sampler_graphs_are_bit_identical).

Completion (NodeAdjEDMSampler.sample_completion) adds one fixed buffer pair, K = the NaN-coded known state, allocated on
the first completion run and refilled per run like X; its graphs (keyed apart from the unconditioned ones) run the
pre-step that reads K and, on the last step, X = apply_known(euler(XH, D1), K) [+ decode].
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from ... import native


class HeunGraphPlan:
    def __init__(self, net, nat, batch: int, n: int, c_e: int, c_n: int, num_steps: int, self_condition: bool,
                 device: torch.device):
        self.net, self.nat = net, nat
        self.key = (id(nat), batch, n, c_e, c_n, num_steps, bool(self_condition))
        self.B, self.N, self.ce, self.cn, self.num_steps = batch, n, c_e, c_n, num_steps
        self.self_condition = bool(self_condition)
        self.dev = device
        self.lib = native.lib()
        f32 = dict(dtype=torch.float32, device=device)

        def pair():
            return torch.zeros(batch, c_e, n, n, **f32), torch.zeros(batch, n, c_n, **f32)

        self.X, self.XH, self.D1, self.SC, self.T = pair(), pair(), pair(), pair(), pair()
        self.K = None   # known state of completion runs (set_known)
        self.flags = torch.zeros(batch, n, dtype=torch.bool, device=device)
        self.table = torch.zeros(num_steps * native.STEP_PARAMS_BYTES, dtype=torch.uint8, device=device)
        self.cur = torch.zeros(native.STEP_PARAMS_BYTES, dtype=torch.uint8, device=device)
        self.counter = torch.zeros(1, dtype=torch.int32, device=device)
        # a float32 view of cur.t_hat: the sigma pointer of the captured denoiser calls
        self.sigma = self.cur[native.STEP_PARAMS_T_HAT_OFFSET:native.STEP_PARAMS_T_HAT_OFFSET + 4].view(torch.float32)
        self.adj_cls = torch.zeros(batch, n, n, dtype=torch.int32, device=device)
        self.node_cls = torch.zeros(batch, n, dtype=torch.int32, device=device)
        self.bbox = torch.zeros(batch, n, 4, **f32)
        self.grid_a, self.inc_a = native.aten_normal_policy(self.X[0].numel(), device)
        self.grid_n, self.inc_n = native.aten_normal_policy(self.X[1].numel(), device)
        # padding skipping: the table is a fixed buffer (its address is part of the captured launches), refilled per
        # sampling run; the bucket geometry is baked into launch grids and TMA descriptors, so it keys the graphs
        from ...model.diffusesg.diffusesg import SkipPlan
        self.skip_tables = torch.zeros(SkipPlan.buffer_len(batch, n, max(1, nat.skip_info()[0])), dtype=torch.int32,
                                       device=device)   # two level tables + the row maps
        self.skip = None
        self.graphs: Dict[Tuple, torch.cuda.CUDAGraph] = {}
        self.pool = None
        self.host_table = np.zeros(num_steps, dtype=np.dtype([
            ("noise_coef", "<f4"), ("inv_t_hat", "<f4"), ("h", "<f4"), ("inv_t_prime", "<f4"), ("t_hat", "<f4"),
            ("reserved", "<f4"), ("seed", "<u8"), ("offset_adj", "<u8"), ("offset_node", "<u8")]))
        assert self.host_table.dtype.itemsize == native.STEP_PARAMS_BYTES
        # everything lazily initialised inside the library (function attributes, workspace) happens outside capture
        self.net.denoise_into(nat, self.XH[0], self.XH[1], self.flags, self.sigma, None, None, self.T[0], self.T[1])

    # --------------------------------------------------------------------------------------------------
    def set_flags(self, flags, skip_padding: bool):
        from ...model.diffusesg.diffusesg import SkipPlan
        self.flags.copy_(flags)
        self.skip = SkipPlan.build(self.nat, flags, self.N, out=self.skip_tables) if skip_padding else None
        if len(self.graphs) > 24:   # many distinct compact sizes seen: drop the captured graphs, keep the buffers
            self.graphs.clear()

    def set_known(self, known):
        """Refill K with this run's condition (allocated on the first completion run); None: an unconditioned run."""
        if known is None:
            return
        if self.K is None:
            self.K = (torch.empty_like(self.X[0]), torch.empty_like(self.X[1]))
        self.K[0].copy_(known[0])
        self.K[1].copy_(known[1])

    def begin(self, scalars, seed: int, offset0: int) -> int:
        """Upload the per-step table for one sampling run; returns the generator offset after the run."""
        t = self.host_table
        for i, sc in enumerate(scalars):
            t[i] = (sc["noise_coef"], sc["inv_t_hat"], sc["h"], sc["inv_t_prime"], float(sc["t_hat"]), 0.0, seed,
                    offset0 + i * (self.inc_a + self.inc_n), offset0 + i * (self.inc_a + self.inc_n) + self.inc_a)
        self.table.copy_(torch.from_numpy(t.view(np.uint8).reshape(-1)), non_blocking=False)
        self.counter.zero_()
        return offset0 + len(scalars) * (self.inc_a + self.inc_n)

    def step_offset(self, offset0: int, i: int) -> int:
        return offset0 + i * (self.inc_a + self.inc_n)

    def advance_only(self):
        """Eager steps (profiling) still have to move the table cursor."""
        native.check(self.lib.dsg_edm_step_advance(self.table.data_ptr(), self.cur.data_ptr(), self.counter.data_ptr(),
                                                   native.stream_ptr(self.dev)), "dsg_edm_step_advance")

    # --------------------------------------------------------------------------------------------------
    def _issue(self, c1: bool, c2: bool, last: bool, decode: Optional[Tuple[int, int, bool]], known: bool = False):
        """The launches of one step, on the current stream (called under capture)."""
        lib, st = self.lib, native.stream_ptr(self.dev)
        B, N, ce, cn = self.B, self.N, self.ce, self.cn
        cur = self.cur.data_ptr()
        p = lambda t: t.data_ptr()
        native.check(lib.dsg_edm_step_advance(p(self.table), cur, p(self.counter), st), "dsg_edm_step_advance")
        if known:
            native.check(lib.dsg_edm_pre_step_philox_known(p(self.X[0]), p(self.X[1]), p(self.K[0]), p(self.K[1]),
                                                           p(self.flags), 0.0, 0.0, 0, 0, self.grid_a, 0, self.grid_n, cur,
                                                           p(self.XH[0]), p(self.XH[1]), B, ce, N, cn, st),
                         "dsg_edm_pre_step_philox_known")
        else:
            native.check(lib.dsg_edm_pre_step_philox_dev(p(self.X[0]), p(self.X[1]), p(self.flags), cur, self.grid_a,
                                                         self.grid_n, p(self.XH[0]), p(self.XH[1]), B, ce, N, cn, st),
                         "dsg_edm_pre_step_philox_dev")
        sc = self.SC if self.self_condition else (None, None)

        def D(sc_pair, out):
            self.net.denoise_into(self.nat, self.XH[0], self.XH[1], self.flags, self.sigma, sc_pair[0], sc_pair[1],
                                  out[0], out[1], self.skip)

        if c1:
            D(sc, self.T)
            D(self.T, self.D1)
        else:
            D(sc, self.D1)
        if last and known:
            native.check(lib.dsg_edm_post_step_dev(p(self.XH[0]), p(self.XH[1]), p(self.D1[0]), p(self.D1[1]), None,
                                                   None, p(self.flags), cur, p(self.X[0]), p(self.X[1]), B, ce, N, cn,
                                                   st), "dsg_edm_post_step_dev")
            native.check(lib.dsg_edm_apply_known(p(self.X[0]), p(self.X[1]), p(self.K[0]), p(self.K[1]), p(self.flags),
                                                 B, ce, N, cn, st), "dsg_edm_apply_known")
            if decode is not None:
                native.check(lib.dsg_decode_samples(p(self.X[0]), p(self.X[1]), p(self.flags), p(self.adj_cls),
                                                    p(self.node_cls), p(self.bbox), decode[0], decode[1], B, ce, N, cn,
                                                    st), "dsg_decode_samples")
            return
        if last:
            if decode is None:
                native.check(lib.dsg_edm_post_step_dev(p(self.XH[0]), p(self.XH[1]), p(self.D1[0]), p(self.D1[1]), None,
                                                       None, p(self.flags), cur, p(self.X[0]), p(self.X[1]), B, ce, N,
                                                       cn, st), "dsg_edm_post_step_dev")
            else:
                n_adj, n_node, want_state = decode
                native.check(lib.dsg_edm_final_step_decode(
                    p(self.XH[0]), p(self.XH[1]), p(self.D1[0]), p(self.D1[1]), p(self.flags), 0.0, 0.0, cur,
                    p(self.X[0]) if want_state else None, p(self.X[1]) if want_state else None, p(self.adj_cls),
                    p(self.node_cls), p(self.bbox), n_adj, n_node, B, ce, N, cn, st), "dsg_edm_final_step_decode")
            return
        sc2 = self.D1 if self.self_condition else (None, None)
        if c2:
            D(sc2, self.T)
            D(self.T, self.SC)
        else:
            D(sc2, self.SC)
        native.check(lib.dsg_edm_post_step_dev(p(self.XH[0]), p(self.XH[1]), p(self.D1[0]), p(self.D1[1]), p(self.SC[0]),
                                               p(self.SC[1]), p(self.flags), cur, p(self.X[0]), p(self.X[1]), B, ce, N,
                                               cn, st), "dsg_edm_post_step_dev")

    def replay(self, c1: bool, c2: bool, last: bool, decode=None, known: bool = False):
        key = (bool(c1), bool(c2) and not last, bool(last), decode, self.skip.key if self.skip is not None else None,
               bool(known))
        g = self.graphs.get(key)
        if g is None:
            g = torch.cuda.CUDAGraph()
            n0 = native.launch_count()
            with torch.cuda.graph(g, pool=self.pool):
                self._issue(key[0], key[1], key[2], decode, key[5])
            if self.pool is None:
                self.pool = g.pool()
            g.dsg_launches = native.launch_count() - n0   # kernels per replay (counted at capture, nothing ran)
            self.lib.dsg_launch_count_add(C.c_uint64(-g.dsg_launches & (2 ** 64 - 1)))
            self.graphs[key] = g
        g.replay()
        self.lib.dsg_launch_count_add(g.dsg_launches)
        return (1 + int(key[0])) + (0 if last else 1 + int(key[1]))   # raw denoiser passes of the step
