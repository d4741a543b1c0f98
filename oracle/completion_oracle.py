"""CPU oracle for scene-graph completion (TEST INFRASTRUCTURE ONLY).

The EDM stochastic-Heun loop of ``edm_oracle`` with a set of state entries held at known clean values
(``NodeAdjEDMSampler.sample_completion``, DESIGN.md §3.6).  ``known = (known_adj, known_node)`` has the shapes of the
state; a finite value is a known entry, NaN a free one.  Step i of ``edm_oracle.heun_step`` changes in two places:

* pre-step, with the same eps at the same element:  x_hat = mask(isnan(k) ? x + noise_coef * eps : k + t_hat * eps)
* after the last (Euler) update:                    x     = mask(isnan(k) ? x : k)

Everything else - scalars, denoiser calls, self-conditioning, the Heun update, the order in which ``normal`` is
called - is ``edm_oracle``'s, so an all-NaN ``known`` gives ``edm_oracle.sample`` bit for bit
(tests/test_completion_host.py).
"""
from __future__ import annotations

from typing import Callable, Optional

import torch

from . import edm_oracle as E
from .denoiser_oracle import mask_pairs, mask_rows

Tensor = torch.Tensor


def heun_step(model, adjs, nodes, flags, sc_a, sc_n, t_cur, t_next, i, num_steps, normal: Callable, known,
              self_condition: bool = True, gt=None):
    """edm_oracle.heun_step with the two completion rules; returns (adjs_next, nodes_next, sc_a, sc_n)."""
    s = E.step_scalars(t_cur, t_next, num_steps)
    t_hat, h, t_prime = s["t_hat"], s["h"], s["t_prime"]
    eps = normal(tuple(adjs.shape))
    adjs_hat = mask_pairs(torch.where(known[0].isnan(), adjs + s["noise_coef"] * eps, known[0] + t_hat * eps), flags)
    eps = normal(tuple(nodes.shape))
    nodes_hat = mask_rows(torch.where(known[1].isnan(), nodes + s["noise_coef"] * eps, known[1] + t_hat * eps), flags)
    sig = t_hat.view(-1).expand(flags.size(0))

    def denoise(sa, sn):
        if gt is not None:
            return gt
        da, dn = model(adjs_hat, nodes_hat, flags, sig, sa, sn)
        return mask_pairs(da, flags), mask_rows(dn, flags)

    d1a, d1n = denoise(sc_a, sc_n)
    inv = 1.0 / t_hat
    k_a = mask_pairs(inv * adjs_hat - inv * d1a, flags)
    k_n = mask_rows(inv * nodes_hat - inv * d1n, flags)
    prime_a = adjs_hat + h * k_a
    prime_n = nodes_hat + h * k_n
    if i == num_steps - 1:
        next_a, next_n = prime_a, prime_n
        da, dn = d1a, d1n
    else:
        if gt is None and self_condition:
            sc_a, sc_n = d1a, d1n
        da, dn = denoise(sc_a, sc_n)
        inv_p = 1.0 / t_prime
        kp_a = inv_p * prime_a - inv_p * da
        kp_n = inv_p * prime_n - inv_p * dn
        next_a = adjs_hat + h * (0.5 * k_a + 0.5 * kp_a)
        next_n = nodes_hat + h * (0.5 * k_n + 0.5 * kp_n)
    next_a, next_n = mask_pairs(next_a, flags), mask_rows(next_n, flags)
    if i == num_steps - 1:
        next_a = mask_pairs(torch.where(known[0].isnan(), next_a, known[0]), flags)
        next_n = mask_rows(torch.where(known[1].isnan(), next_n, known[1]), flags)
    if self_condition:
        sc_a, sc_n = da, dn
    return next_a, next_n, sc_a, sc_n


def sample(model, flags: Tensor, c_e: int, c_n: int, known, num_steps: int = E.NUM_STEPS,
           normal: Optional[Callable] = None, self_condition: bool = True, gt=None):
    """edm_oracle.sample with ``known`` held; returns the final (adjs, nodes)."""
    if normal is None:
        normal = lambda shape: torch.randn(shape)
    ts = E.t_steps_fp32(num_steps)
    adjs, nodes = E.init_sample(flags, c_e, c_n, normal)
    adjs, nodes = adjs * ts[0], nodes * ts[0]
    sc_a = sc_n = None
    for i in range(num_steps):
        adjs, nodes, sc_a, sc_n = heun_step(model, adjs, nodes, flags, sc_a, sc_n, ts[i], ts[i + 1], i, num_steps,
                                            normal, known, self_condition, gt)
    return adjs, nodes


def encode_known(flags: Tensor, c_e: int, c_n: int, node_cls=None, bbox=None, adj_cls=None):
    """Conditions -> NaN-coded (known_adj [B,c_e,N,N], known_node [B,N,c_n]): the inverse of edm_oracle.decode_samples
    for the 'bits' encodings.  A known class (>= 0; -1 = free) becomes its bits, MSB first, as +-1; a box coordinate b
    (NaN = free) becomes 2 b - 1."""
    b, n = flags.shape
    nb = c_n - 4
    known_adj = torch.full((b, c_e, n, n), float("nan"))
    known_node = torch.full((b, n, c_n), float("nan"))

    def bits(cls, width):   # int [...] -> [..., width] of +-1.0, MSB first
        shifts = torch.arange(width - 1, -1, -1)
        return ((cls.long()[..., None] >> shifts) & 1).float() * 2.0 - 1.0

    if adj_cls is not None:
        on = adj_cls >= 0
        known_adj = torch.where(on[:, None], bits(adj_cls.clamp_min(0), c_e).permute(0, 3, 1, 2), known_adj)
    if node_cls is not None:
        on = node_cls >= 0
        known_node[..., :nb] = torch.where(on[..., None], bits(node_cls.clamp_min(0), nb), known_node[..., :nb])
    if bbox is not None:
        known_node[..., nb:] = 2.0 * bbox.float() - 1.0
    return known_adj, known_node
