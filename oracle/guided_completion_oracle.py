"""CPU oracle for reconstruction-guided scene-graph completion (TEST INFRASTRUCTURE ONLY).

``NodeAdjEDMSampler.sample_completion(..., guidance_scale=w)`` (DESIGN.md §3.7): the completion loop of
``completion_oracle`` in which every denoiser call at x_hat returns

    D~ = mask(D - w grad_x_hat 1/2 sum_known (D(x_hat) - k)^2)

instead of D, computed by fp32 autograd through ``model`` with the self-conditioning inputs held constant.  D~ then
replaces D everywhere downstream (Heun update, self-conditioning hand-off); the pre-step replacement, ``x = k`` after the
last step and the order in which ``normal`` is called are ``completion_oracle``'s.  A model that refreshes its own
self-conditioning (the coin flip) must run that pass under ``torch.no_grad()``, as ``NodeAdjPrecond.forward`` does.

The loop itself is not restated: ``sample`` runs ``completion_oracle.sample`` with the guided denoiser in place of
``model`` (its masks are idempotent on D~), and ``guidance = 0`` is ``completion_oracle.sample`` itself.
"""
from __future__ import annotations

from typing import Callable, Optional

import torch

from . import completion_oracle as CO
from . import edm_oracle as E
from .denoiser_oracle import mask_pairs, mask_rows

Tensor = torch.Tensor


def guided(model, adjs_hat, nodes_hat, flags, sig, sa, sn, known, w: float):
    """mask(D - w grad_x 1/2 sum_known (D(x) - k)^2) at x = (adjs_hat, nodes_hat), fp32 autograd."""
    xa = adjs_hat.detach().requires_grad_(True)
    xn = nodes_hat.detach().requires_grad_(True)
    sa = None if sa is None else sa.detach()
    sn = None if sn is None else sn.detach()
    with torch.enable_grad():
        da, dn = model(xa, xn, flags, sig, sa, sn)
        da, dn = mask_pairs(da, flags), mask_rows(dn, flags)
        ka, kn = known
        ra = torch.where(ka.isnan(), torch.zeros_like(da), da - torch.nan_to_num(ka))
        rn = torch.where(kn.isnan(), torch.zeros_like(dn), dn - torch.nan_to_num(kn))
        loss = 0.5 * (ra.pow(2).sum() + rn.pow(2).sum())
        ga, gn = torch.autograd.grad(loss, (xa, xn))
    return mask_pairs(da.detach() - w * ga, flags), mask_rows(dn.detach() - w * gn, flags)


def sample(model, flags: Tensor, c_e: int, c_n: int, known, num_steps: int = E.NUM_STEPS,
           normal: Optional[Callable] = None, self_condition: bool = True, guidance: float = 0.0):
    """completion_oracle.sample with reconstruction guidance of scale ``guidance``; returns the final (adjs, nodes)."""
    if guidance == 0.0:
        return CO.sample(model, flags, c_e, c_n, known, num_steps=num_steps, normal=normal, self_condition=self_condition)

    def guided_model(adjs_hat, nodes_hat, f, sig, sa, sn):
        return guided(model, adjs_hat, nodes_hat, f, sig, sa, sn, known, guidance)

    return CO.sample(guided_model, flags, c_e, c_n, known, num_steps=num_steps, normal=normal,
                     self_condition=self_condition)
