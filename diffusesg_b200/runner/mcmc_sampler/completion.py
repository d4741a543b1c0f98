"""Conditions for scene-graph completion: user-level known classes and boxes -> the NaN-coded known state.

``NodeAdjEDMSampler.sample_completion`` holds a set of entries of the ``adj [B, C_e, N, N]`` / ``node [B, N, C_n]``
state at given clean values while the sampler draws the others.  Its input is that state with NaN on every free entry
(DESIGN.md §3.6).  ``encode_known`` builds it from what a user usually holds:

* layout from a scene graph: ``node_cls`` and ``adj_cls`` known, ``bbox`` free;
* relation prediction: ``node_cls`` and ``bbox`` known, ``adj_cls`` free;
* object completion: some of each known, the rest free.

Encoding is the inverse of the 'bits' decode (``NodeAdjEDMSampler.sample_decoded``): a class becomes its bits, MSB
first, as +1 / -1 (the first C_n - 4 node channels, or all C_e channels of a pair), a box coordinate b in [0, 1]
becomes 2 b - 1 (the last four node channels) - the encoding of the training data.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from ... import native


def _check_shape(name, t, shape):
    if tuple(t.shape) != tuple(shape):
        raise ValueError(f"{name}: shape {tuple(t.shape)}, expected {tuple(shape)}")


def _check_classes(name, cls, num_type, bits):
    if cls.dtype.is_floating_point or cls.dtype == torch.bool:
        raise ValueError(f"{name}: integer class ids expected (-1 = free), got {cls.dtype}")
    limit = 2 ** bits
    if num_type is not None:
        if not 1 <= int(num_type) <= limit:
            raise ValueError(f"{name}: {num_type} types do not fit {bits} bits")
        limit = int(num_type)
    bad = (cls < -1) | (cls >= limit)
    if bool(bad.any()):
        raise ValueError(f"{name}: class {int(cls[bad][0])} outside [0, {limit}) (use -1 for a free entry)")


def validate_conditions(node_flags, num_edge_chan: int, num_node_chan: int, node_cls=None, bbox=None, adj_cls=None,
                        num_adj_type: Optional[int] = None, num_node_type: Optional[int] = None) -> None:
    """Raise ValueError for any condition encode_known cannot represent or the sampler cannot hold."""
    if node_flags.dim() != 2:
        raise ValueError(f"node_flags: shape {tuple(node_flags.shape)}, expected [B, N]")
    b, n = node_flags.shape
    if not 1 <= num_edge_chan <= 30 or not 5 <= num_node_chan <= 34:
        raise ValueError(f"channels: num_edge_chan {num_edge_chan} must be in [1, 30], num_node_chan {num_node_chan} "
                         "in [5, 34] (class bits + 4 box coordinates)")
    flags = node_flags.bool().cpu()
    if node_cls is not None:
        _check_shape("node_cls", node_cls, (b, n))
        node_cls = node_cls.cpu()
        _check_classes("node_cls", node_cls, num_node_type, num_node_chan - 4)
        if bool(((node_cls >= 0) & ~flags).any()):
            raise ValueError("node_cls: a known class on a node whose flag is 0")
    if bbox is not None:
        _check_shape("bbox", bbox, (b, n, 4))
        if not bbox.dtype.is_floating_point:
            raise ValueError(f"bbox: floating-point boxes expected, got {bbox.dtype}")
        bbox = bbox.cpu().double()
        free_row = bbox.isnan().all(-1)
        known = ~free_row
        if not bool(torch.isfinite(bbox[known]).all()):
            raise ValueError("bbox: a row must be all NaN (free) or all finite")
        if bool(((bbox[known] < 0) | (bbox[known] > 1)).any()):
            raise ValueError("bbox: box coordinates must lie in [0, 1]")
        if bool((known & ~flags).any()):
            raise ValueError("bbox: a known box on a node whose flag is 0")
    if adj_cls is not None:
        _check_shape("adj_cls", adj_cls, (b, n, n))
        adj_cls = adj_cls.cpu()
        _check_classes("adj_cls", adj_cls, num_adj_type, num_edge_chan)
        on = adj_cls >= 0
        if bool(on.diagonal(dim1=1, dim2=2).any()):
            raise ValueError("adj_cls: a known relation on a self-pair (i, i)")
        if bool((on & ~(flags[:, :, None] & flags[:, None, :])).any()):
            raise ValueError("adj_cls: a known relation on a pair with a node whose flag is 0")


def encode_known(node_flags, num_edge_chan: int, num_node_chan: int, node_cls=None, bbox=None, adj_cls=None,
                 num_adj_type: Optional[int] = None, num_node_type: Optional[int] = None
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
    """``(known_adj [B, C_e, N, N], known_node [B, N, C_n])`` fp32 on the device of ``node_flags`` (the current CUDA
    device for host flags), NaN on every free entry, for ``NodeAdjEDMSampler.sample_completion``.

    ``node_cls [B, N]`` / ``adj_cls [B, N, N]``: integer class ids, -1 = free; ``bbox [B, N, 4]``: boxes in [0, 1], a
    row of NaN = free.  Any of them may be None (all free).  ``num_node_type`` / ``num_adj_type`` bound the classes
    (default: what the channel bits can hold).  Every input is checked before any kernel runs (ValueError)."""
    validate_conditions(node_flags, num_edge_chan, num_node_chan, node_cls, bbox, adj_cls, num_adj_type, num_node_type)
    b, n = node_flags.shape
    dev = node_flags.device if node_flags.is_cuda else torch.device("cuda", torch.cuda.current_device())
    i32 = lambda t: None if t is None else t.to(device=dev, dtype=torch.int32).contiguous()
    box = None if bbox is None else bbox.to(device=dev, dtype=torch.float32).contiguous()
    return native.encode_known(i32(node_cls), box, i32(adj_cls), b, num_edge_chan, n, num_node_chan, dev)
