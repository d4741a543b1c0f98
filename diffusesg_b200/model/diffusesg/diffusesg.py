"""Drop-in ``DiffuseSG`` denoiser backed by libdsg_b200 (hand-written sm_100a CUDA).

Mirrors the reference interface (model/diffusesg/diffusesg.py:587-830 of ubc-vision/DiffuseSG):

* the same constructor keywords as used by ``get_network`` (utils/learning_utils.py:47-64);
* the same ``state_dict()`` keys, order, shapes and dtypes (247 entries for the Visual Genome config,
  including the persistent ``relative_position_index`` / ``attn_mask`` buffers), so reference checkpoints load
  with ``strict=True`` and ``ema_pytorch.EMA`` / DDP can wrap the module;
* ``forward(adj, node, node_flags, noise_labels, self_cond_x=None, self_cond_feat=None) -> (adj_out, node_out)``.

The module holds ordinary fp32 ``nn.Parameter`` masters.  The native side keeps its own arena with the packed
bf16 / transposed / folded copies; it is refreshed lazily whenever a parameter changed (version counters, plus a
device-side comparison with the arena's master copies that also catches writes through ``.data``).  There
is no PyTorch implementation of the forward in this file: without the shared library or a CUDA device the call
raises.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence

import torch
import torch.nn as nn

from ... import native
from .geometry import relative_position_index, shifted_window_mask


class _Tree(nn.Module):
    """Anonymous container node: gives parameters the dotted names of the reference module tree."""


def _spec(img: int, cin: int, embed: int, depths: Sequence[int], heads: Sequence[int], window: int, c_e: int, c_n: int):
    """Ordered [(key, shape, kind)] in the registration order of the reference (diffusesg.py:611-720)."""
    out: List[tuple] = []

    def lin(p, o, i, bias=True, kind="w"):
        out.append((p + ".weight", (o, i), kind))
        if bias:
            out.append((p + ".bias", (o,), "zero"))

    def ln(p, c):
        out.append((p + ".weight", (c,), "one"))
        out.append((p + ".bias", (c,), "zero"))

    def block(p, dim, res, nh, j):
        w, s = (res, 0) if res <= window else (window, 0 if j % 2 == 0 else window // 2)
        if s > 0:
            out.append((p + ".attn_mask", ((res // w) ** 2, w * w, w * w), ("mask", res, w, s)))
        lin(p + ".affine", 2 * dim, 512)
        ln(p + ".norm1", dim)
        out.append((p + ".attn.relative_position_bias_table", ((2 * w - 1) ** 2, nh), "table"))
        out.append((p + ".attn.relative_position_index", (w * w, w * w), ("index", w)))
        lin(p + ".attn.qkv", 3 * dim, dim)
        lin(p + ".attn.proj", dim, dim)
        ln(p + ".norm2", dim)
        lin(p + ".mlp.fc1", 4 * dim, dim)
        lin(p + ".mlp.fc2", dim, 4 * dim)

    nl = len(depths)
    lin("patch_embed.affine", 2 * embed, 512)
    out.append(("patch_embed.proj.weight", (embed, cin, 1, 1), "conv"))
    out.append(("patch_embed.proj.bias", (embed,), ("conv_bias", cin)))
    ln("patch_embed.norm", embed)
    for s in range(nl):
        dim, res = embed * 2 ** s, img // 2 ** s
        for j in range(depths[s]):
            block(f"down_layers.{s}.blocks.{j}", dim, res, heads[s], j)
        if s < nl - 1:
            lin(f"down_layers.{s}.downsample.reduction", 2 * dim, 4 * dim, bias=False)
            ln(f"down_layers.{s}.downsample.norm", 4 * dim)
    for u in range(nl):
        s = nl - 1 - u
        dim, res = embed * 2 ** s, img // 2 ** s
        if u > 0:
            d = 4 * dim
            lin(f"up_layers.{u}.upsample.pre_linear", d, d, bias=False)
            ln(f"up_layers.{u}.upsample.norm", d)
            lin(f"up_layers.{u}.upsample.post_linear", d // 4, d // 4, bias=False)
            ln(f"up_layers.{u}.upsample.post_norm", d // 4)
        for j in range(depths[s]):
            block(f"up_layers.{u}.blocks.{j}", dim, res, heads[s], j)
    for k in range(3):
        out.append((f"read_out.{k}.weight", (embed, embed, 1, 1), "conv"))
        out.append((f"read_out.{k}.bias", (embed,), ("conv_bias", embed)))
    lin("map_layer0", 512, embed)
    lin("map_layer1", 512, 512)
    ln("norm", embed)
    lin("readout_adj_mlp.fc1", embed, embed)
    lin("readout_adj_mlp.fc2", c_e, embed)
    lin("readout_node_mlp.fc1", embed, embed)
    lin("readout_node_mlp.fc2", c_n, embed)
    return out


class DiffuseSG(nn.Module):
    def __init__(self, img_size=224, patch_size=4, in_chans=3, embed_dim=96, depths=(2, 2, 6, 2),
                 num_heads=(3, 6, 12, 24), window_size=7, mlp_ratio=4., qkv_bias=True, qk_scale=None, drop_rate=0.,
                 attn_drop_rate=0., drop_path_rate=0.1, out_chans_adj=1, out_chans_node=1, norm_layer=nn.LayerNorm,
                 patch_norm=True, use_checkpoint=False, self_condition=False, symmetric_noise=True, **kwargs):
        super().__init__()
        img_size = int(img_size[0] if isinstance(img_size, (tuple, list)) else img_size)
        unsupported = []
        if int(patch_size) != 1:
            unsupported.append(f"patch_size={patch_size} (the scene-graph configs use 1)")
        if float(mlp_ratio) != 4.0:
            unsupported.append(f"mlp_ratio={mlp_ratio}")
        if not qkv_bias or qk_scale is not None or not patch_norm or norm_layer is not nn.LayerNorm:
            unsupported.append("non-default qkv_bias / qk_scale / patch_norm / norm_layer")
        if drop_rate or attn_drop_rate or drop_path_rate:
            unsupported.append("non-zero dropout / stochastic depth (get_network passes 0 for all three)")
        if symmetric_noise:
            unsupported.append("symmetric_noise=True (scene graphs use non-symmetric noise, learning_utils.py:62)")
        if unsupported:
            raise NotImplementedError("DiffuseSG (B200): " + "; ".join(unsupported))
        depths, num_heads = list(depths), list(num_heads)[:len(depths)]
        self.num_layers = len(depths)
        self.embed_dim = int(embed_dim)
        self.img_size = img_size
        self.depths, self.num_heads, self.window_size = depths, num_heads, int(window_size)
        self.self_condition = bool(self_condition)
        self.symmetric_noise = False
        self.out_chans_adj, self.out_chans_node = int(out_chans_adj), int(out_chans_node)
        self.num_features = int(embed_dim * 2 ** (self.num_layers - 1))
        self.mlp_ratio = mlp_ratio
        self.patches_resolution = [img_size, img_size]
        cin = in_chans * 2 if self_condition else in_chans
        if cin != (self.out_chans_adj + 2 * self.out_chans_node) * (2 if self_condition else 1):
            raise NotImplementedError(f"in_chans={in_chans} is not out_chans_adj + 2 * out_chans_node "
                                      "(utils/sg_utils.py:412-430 always builds it that way)")
        self._spec = _spec(img_size, cin, self.embed_dim, depths, num_heads, self.window_size, self.out_chans_adj,
                           self.out_chans_node)
        for key, shape, kind in self._spec:
            *path, leaf = key.split(".")
            node = self
            for name in path:
                node = DiffuseSG._child(node, name)
            if isinstance(kind, tuple) and kind[0] == "index":
                node.register_buffer(leaf, relative_position_index(kind[1]))
            elif isinstance(kind, tuple) and kind[0] == "mask":
                node.register_buffer(leaf, shifted_window_mask(kind[1], kind[2], kind[3]))
            else:
                node.register_parameter(leaf, nn.Parameter(self._init(shape, kind)))
        # native state (never part of state_dict, never deep-copied)
        self.__dict__["_nat"] = None

    @staticmethod
    def _child(module: nn.Module, name: str) -> _Tree:
        if name not in module._modules:
            module.add_module(name, _Tree())
        return module._modules[name]

    @staticmethod
    def _init(shape, kind) -> torch.Tensor:
        """Same distributions as the reference init (diffusesg.py:722-729 and nn.Conv2d defaults)."""
        t = torch.empty(shape)
        if kind in ("w", "table"):
            nn.init.trunc_normal_(t, std=.02)
        elif kind == "zero":
            t.zero_()
        elif kind == "one":
            t.fill_(1.0)
        elif kind == "conv":
            nn.init.kaiming_uniform_(t, a=math.sqrt(5))
        elif isinstance(kind, tuple) and kind[0] == "conv_bias":
            bound = 1 / math.sqrt(kind[1])
            nn.init.uniform_(t, -bound, bound)
        else:  # pragma: no cover
            raise AssertionError(kind)
        return t

    # ------------------------------------------------------------------------------------------------------
    # native model management
    # ------------------------------------------------------------------------------------------------------
    def __deepcopy__(self, memo):
        # ema_pytorch.EMA deep-copies the online model (utils/learning_utils.py:160): copy the parameters,
        # give the copy its own (lazily created) native state
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        import copy
        for k, v in self.__dict__.items():
            if k in ("_nat", "_train_state", "_active_skip"):   # device-side state is rebuilt lazily by the copy
                new.__dict__[k] = None
            else:
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    def __getstate__(self):
        d = dict(self.__dict__)
        d["_nat"] = None
        d.pop("_train_state", None)
        d.pop("_active_skip", None)
        return d

    def _versions(self):
        # (version counter, storage address) of every parameter / buffer: moves on optimizer steps,
        # load_state_dict and .to(device).  NOT on writes through `.data` (ema_pytorch's `.data.lerp_()`,
        # `p.data.copy_()`): those are caught by the deep probe below.
        return tuple((t._version, t.data_ptr()) for t in self.state_dict(keep_vars=True).values())

    def _native(self, device: torch.device) -> "_NativeModel":
        """The native model for `device`, with its weight arena brought up to date.

        Staleness is detected in two tiers: autograd version counters / storage addresses (free), and - because
        writes through `.data` leave those untouched - a device-side comparison of every parameter with the fp32
        master the arena holds (`dsg_model_tensor_differs`: one small launch per tensor and one 4-byte readback).
        Inside `frozen_weights()` (the sampler wraps its loop in it) both tiers are skipped after the first call."""
        nat = self.__dict__.get("_nat")
        if nat is None or nat.device != device:
            nat = _NativeModel(self, device)
            self.__dict__["_nat"] = nat
        if self.__dict__.get("_frozen", 0) > 0 and nat.versions is not None and self.__dict__.get("_frozen_checked"):
            return nat
        state = self.state_dict(keep_vars=True)
        ver = tuple((t._version, t.data_ptr()) for t in state.values())
        if nat.versions != ver or nat.differs(state):
            nat.upload(state)
            nat.versions = ver
        self.__dict__["_frozen_checked"] = True
        return nat

    def invalidate_native(self) -> None:
        """Force a re-upload of the weights on the next call."""
        nat = self.__dict__.get("_nat")
        if nat is not None:
            nat.versions = None

    def frozen_weights(self):
        """Context manager: the caller promises not to modify the parameters inside (the EDM sampling loop); the
        staleness checks then run once, on the first call inside the context."""
        return _Frozen(self)

    def train(self, mode: bool = True):
        # train()/eval() transitions are where training loops hand the weights over for sampling
        self.__dict__["_frozen_checked"] = False
        return super().train(mode)

    def forward(self, adj, node, node_flags, noise_labels, self_cond_x=None, self_cond_feat=None):
        """Raw network F(adj, node | node_flags, c_noise)  (reference diffusesg.py:765-830).

        adj [B, C_e, N, N], node [B, N, C_n], node_flags [B, N] bool, noise_labels [B] (or a stride-0 expand of
        one value) -> (adj_out [B, C_e, N, N], node_out [B, N, C_n]), fp32, masked like the reference.
        """
        return self._run(0, adj, node, node_flags, noise_labels, self_cond_x, self_cond_feat)

    def denoise(self, adjs, nodes, node_flags, sigmas, self_cond_adjs=None, self_cond_nodes=None):
        """EDM-preconditioned call D(x; sigma) = mask(c_skip x + c_out F(c_in x, ln(sigma)/4, self_cond)):
        the body of NodeAdjPrecond.forward after the coin flip (model/precond/precond.py:100-105) in one
        native schedule (the scalings ride inside the patch-embedding and read-out kernels)."""
        return self._run(1, adjs, nodes, node_flags, sigmas, self_cond_adjs, self_cond_nodes)

    def denoise_into(self, nat, adjs, nodes, flags, sigma_ptr_tensor, sc_adjs, sc_nodes, out_adjs, out_nodes, skip=None):
        """`denoise` on pre-validated contiguous fp32 CUDA tensors with one shared sigma read from device memory and
        caller-provided outputs: no allocation, no checks - what the sampler captures into its CUDA graphs."""
        nat.forward(1, adjs.shape[0], 1, adjs, nodes, flags, sigma_ptr_tensor, 0, sc_adjs, sc_nodes, out_adjs, out_nodes,
                    skip)

    def make_skip_plan(self, node_flags, device=None, force=False):
        """Padded-row skipping plan for a batch with these node flags (include/dsg_b200.h: dsg_model_skip_info), or
        None when the geometry has no compactable stage or the batch has (almost) no padding to skip.  Reads the
        flags on the host (one small D2H copy): build it once per batch, not per call."""
        device = torch.device(device) if device is not None else node_flags.device
        return SkipPlan.build(self._native(device), node_flags, self.img_size, min_saving=-1e9 if force else 0.03)

    def skipping(self, plan):
        """Context manager: calls with one shared noise level and the plan's batch size inside use `plan`."""
        return _Skipping(self, plan)

    def _run(self, mode, adj, node, flags, noise, sc_adj, sc_node):
        grad = torch.is_grad_enabled()
        params = grad and self.training and any(p.requires_grad for p in self.parameters())
        # an input that requires grad runs the tape too (eval mode included): adj / node get their gradients, the noise
        # levels and self-conditioning inputs raise NotImplementedError in backward
        inputs = grad and any(isinstance(t, torch.Tensor) and t.requires_grad for t in (adj, node, noise, sc_adj, sc_node))
        train = params or inputs
        if not train and self.training and not grad and self.__dict__.get("_train_state") is not None:
            train = True    # no-grad pass inside a training loop (self-conditioning refresh): the training kernels, no tape
        if adj.dim() != 4 or node.dim() != 3 or flags.dim() != 2:
            raise NotImplementedError("DiffuseSG (B200): expects adj [B,C,N,N], node [B,N,C], node_flags [B,N] "
                                      "(the scene-graph path of the reference)")
        dev = adj.device
        adj = native.require_cuda(adj, "adj")
        node = native.require_cuda(node.to(dev), "node")
        b, ce, n, _ = adj.shape
        if (ce, n, node.shape[-1]) != (self.out_chans_adj, self.img_size, self.out_chans_node):
            raise ValueError(f"input shapes {tuple(adj.shape)}, {tuple(node.shape)} do not match the model "
                             f"(C_e={self.out_chans_adj}, N={self.img_size}, C_n={self.out_chans_node})")
        flags = native.require_cuda(flags.to(dev), "node_flags", torch.bool)
        noise = noise.to(dev)
        if noise.dim() == 0:
            noise = noise.view(1)
        if noise.dtype != torch.float32:
            noise = noise.float()
        if noise.numel() == 1 or (noise.dim() == 1 and noise.stride(0) == 0):
            n_cond, stride = 1, 0
        else:
            if noise.numel() != b:
                raise ValueError(f"noise conditioning has {noise.numel()} entries for batch {b}")
            noise = noise.reshape(b)
            n_cond, stride = b, noise.stride(0)
        if self.self_condition:
            sc_adj = None if sc_adj is None else native.require_cuda(sc_adj, "self_cond_x")
            sc_node = None if sc_node is None else native.require_cuda(sc_node, "self_cond_feat")
        else:
            sc_adj = sc_node = None
        if train:
            # training step (SURVEY 8 f-2): forward with saved activations as one autograd node, model/diffusesg/train_graph.py
            from .train_graph import run_training_forward
            noise_b = (noise.reshape(-1)[:1].expand(b) if n_cond == 1 else noise).contiguous()   # one value or a stride-0 expand
            return run_training_forward(self, mode, adj, node, flags, noise_b, sc_adj, sc_node, params=params)
        nat = self._native(dev)
        out_adj = torch.empty_like(adj)
        out_node = torch.empty_like(node)
        skip = self.__dict__.get("_active_skip")
        if skip is not None and (n_cond != 1 or skip.batch != b or skip.nat is not nat):
            skip = None
        nat.forward(mode, b, n_cond, adj, node, flags, noise, stride, sc_adj, sc_node, out_adj, out_node, skip)
        return out_adj, out_node


class SkipPlan:
    """Compact layout of the padding skipping for one batch of node flags (include/dsg_b200.h: dsg_model_skip_info):
    device table ``perm | tok0 | width`` (int32) plus the bucket geometry that goes into ``dsg_forward_args``."""

    TABLE_EXTRA = 17   # phantom + one dummy image per bucket (<= 8 buckets)

    def __init__(self, nat, batch, tables, n_images_cap, counts, sides, phantom_tok0, kept_fraction, level2=None):
        self.nat, self.batch, self.tables, self.n_images_cap = nat, batch, tables, n_images_cap
        self.counts, self.sides, self.phantom_tok0, self.kept_fraction = counts, sides, phantom_tok0, kept_fraction
        # level2: (table offset in `tables`, counts, sides, phantom_tok0, kept fraction) of the second, coarser layout
        self.level2 = level2
        # what the launch sequence of a pass depends on
        self.key = (tuple(counts), tuple(sides), phantom_tok0) + ((tuple(level2[1]), tuple(level2[2]), level2[3]) if level2 else ())

    @staticmethod
    def table_len(batch: int) -> int:
        """int32 entries of one level's table; the device buffer holds two levels back to back, then the row maps."""
        return (batch + SkipPlan.TABLE_EXTRA) + 2 * batch

    @staticmethod
    def buffer_len(batch: int, n: int, stages: int) -> int:
        """int32 entries of the whole device buffer: two level tables + up to three row maps at the first dense stage
        (dense grid: B res^2 tokens; a compact layout never holds more than (B + 1) res^2)."""
        res = n >> stages
        return 2 * SkipPlan.table_len(batch) + (3 * batch + 2) * res * res

    @staticmethod
    def corner_index(tok0, width, sh, b, res):
        """[res, res] int64: index of token (r, x) of sample b in a compact layout at stage `sh`, -1 outside its corner."""
        import numpy as np
        wc = int(width[b]) >> sh
        idx = np.full((res, res), -1, dtype=np.int64)
        rr, xx = np.meshgrid(np.arange(wc), np.arange(wc), indexing="ij")
        idx[:wc, :wc] = (int(tok0[b]) >> (2 * sh)) + rr * wc + xx
        return idx

    @staticmethod
    def row_maps(table, counts, sides, phantom_tok0, batch, n, stages, level2=None):
        """Row maps of include/dsg_b200.h (dsg_forward_args.skip_map_* / skip2_map_*), as int32 numpy arrays."""
        import numpy as np
        cap = batch + SkipPlan.TABLE_EXTRA
        res = n >> stages
        tok0, width = table[cap:cap + batch], table[cap + batch:cap + 2 * batch]
        ph1 = phantom_tok0 >> (2 * stages)
        c1 = np.stack([SkipPlan.corner_index(tok0, width, stages, b, res) for b in range(batch)])     # [B, res, res]
        if level2 is None:
            return dict(dense_from_c1=np.where(c1 >= 0, c1, ph1).astype(np.int32).reshape(-1))
        table2, counts2, sides2, phantom2_tok0 = level2
        tok2, width2 = table2[cap:cap + batch], table2[cap + batch:cap + 2 * batch]
        perm2 = table2[:sum(counts2)]
        ph2 = phantom2_tok0 >> (2 * stages)
        c2 = np.stack([SkipPlan.corner_index(tok2, width2, stages, b, res) for b in range(batch)])    # [B, res, res]
        dense_from_c2 = np.where(c2 >= 0, c2, ph2).astype(np.int32).reshape(-1)
        c2_from_c1, c2_from_dense = [], []
        img = 0
        for cnt, side in zip(counts2, sides2):
            st = side >> stages
            for k in range(cnt):
                b = int(perm2[img + k])
                if b < 0:
                    c2_from_c1.append(np.full(st * st, ph1, dtype=np.int64))
                    c2_from_dense.append(np.zeros(st * st, dtype=np.int64))
                else:
                    sub = c1[b, :st, :st]
                    c2_from_c1.append(np.where(sub >= 0, sub, ph1).reshape(-1))
                    rr, xx = np.meshgrid(np.arange(st), np.arange(st), indexing="ij")
                    c2_from_dense.append((b * res * res + rr * res + xx).reshape(-1))
            img += cnt
        return dict(c2_from_c1=np.concatenate(c2_from_c1).astype(np.int32), dense_from_c2=dense_from_c2,
                    c2_from_dense=np.concatenate(c2_from_dense).astype(np.int32))

    @staticmethod
    def host_tables(flags_host: torch.Tensor, n: int, granule: int):
        """-> (int32 table, counts, sides, phantom_tok0, compact pixels) or None when more than 8 buckets would be needed."""
        import numpy as np
        f = flags_host.to(torch.bool).cpu().numpy()
        b = f.shape[0]
        last = np.where(f.any(1), n - np.argmax(f[:, ::-1], axis=1), 0)          # index of the last valid node + 1
        rb = np.minimum(n, np.maximum(granule, -(-last // granule) * granule)).astype(np.int64)
        sides = sorted(set(rb.tolist()) | {granule})      # the phantom lives in the bucket of side `granule`
        if len(sides) > 8:
            return None
        cap = b + SkipPlan.TABLE_EXTRA
        table = np.zeros(SkipPlan.table_len(b), dtype=np.int32)
        perm, counts, tok, phantom_tok0 = [], [], 0, 0
        tok0 = np.zeros(b, dtype=np.int64)
        for side in sides:
            members = np.nonzero(rb == side)[0]
            tok0[members] = tok + np.arange(len(members)) * side * side
            images = members.tolist()
            if side == granule:
                phantom_tok0 = tok + len(images) * side * side
                images.append(-1)
            if len(images) % 2:
                images.append(-1)                          # all-padding dummy: the 8 x 8 kernel pairs windows
            perm += images
            counts.append(len(images))
            tok += len(images) * side * side
        table[:len(perm)] = perm
        table[cap:cap + b] = tok0
        table[cap + b:cap + 2 * b] = rb
        return table, counts, sides, int(phantom_tok0), int(tok)

    @staticmethod
    def build(nat, node_flags, n, out=None, min_saving=0.03):
        import numpy as np
        stages, granule = nat.skip_info()
        if stages == 0 or node_flags.dim() != 2 or node_flags.shape[1] != n:
            return None
        b = node_flags.shape[0]
        flags_host = node_flags.to(torch.bool).cpu()
        res = SkipPlan.host_tables(flags_host, n, granule)
        if res is None:
            return None
        table, counts, sides, phantom_tok0, pixels = res
        if pixels > (1.0 - min_saving) * b * n * n and min_saving > -1e8:
            return None      # (almost) nothing to skip: the dense schedule is as fast and has no phantom
        if pixels > (b + 1) * n * n:
            return None      # would not fit the workspace (only possible when forced on a batch without padding)
        level2 = None
        table2 = np.zeros(SkipPlan.table_len(b), dtype=np.int32)
        granule2 = nat.skip_info2()
        if granule2 > 0:
            res2 = SkipPlan.host_tables(flags_host, n, granule2)
            if res2 is not None and res2[4] <= min((b + 1) * n * n, (1.0 - min_saving) * b * n * n if min_saving > -1e8 else 1e30):
                table2, counts2, sides2, phantom2, pixels2 = res2
                level2 = (SkipPlan.table_len(b), counts2, sides2, phantom2, pixels2 / float(b * n * n))
        maps = SkipPlan.row_maps(table, counts, sides, phantom_tok0, b, n, stages,
                                 (table2, level2[1], level2[2], level2[3]) if level2 else None)
        parts, map_offsets, off = [table, table2], {}, 2 * SkipPlan.table_len(b)
        for name, arr in maps.items():
            map_offsets[name] = off
            parts.append(arr)
            off += len(arr)
        t = torch.from_numpy(np.concatenate(parts))
        if out is None:
            out = t.to(nat.device)
        else:
            out[:t.numel()].copy_(t)
        plan = SkipPlan(nat, b, out, b + SkipPlan.TABLE_EXTRA, counts, sides, phantom_tok0, pixels / float(b * n * n), level2)
        plan.map_offsets = map_offsets
        return plan


class _Skipping:
    def __init__(self, module, plan):
        self.m, self.plan = module, plan

    def __enter__(self):
        self.prev = self.m.__dict__.get("_active_skip")
        self.m.__dict__["_active_skip"] = self.plan
        return self.plan

    def __exit__(self, *exc):
        self.m.__dict__["_active_skip"] = self.prev
        return False


class _Frozen:
    def __init__(self, module: "DiffuseSG"):
        self.m = module

    def __enter__(self):
        d = self.m.__dict__
        if d.get("_frozen", 0) == 0:
            d["_frozen_checked"] = False
        d["_frozen"] = d.get("_frozen", 0) + 1
        return self.m

    def __exit__(self, *exc):
        self.m.__dict__["_frozen"] -= 1
        return False


class _NativeModel:
    """Owns the dsg_model handle, its weight arena and the activation workspace (torch tensors = device memory)."""

    def __init__(self, module: DiffuseSG, device: torch.device):
        if device.type != "cuda":
            raise native.NativeError("DiffuseSG (B200) runs on CUDA devices only; there is no CPU fallback")
        self.lib = native.lib()
        self.device = device
        cfg = native.DsgConfig()
        cfg.img_size, cfg.embed_dim, cfg.num_stages = module.img_size, module.embed_dim, module.num_layers
        for i in range(module.num_layers):
            cfg.depths[i] = module.depths[i]
            cfg.num_heads[i] = module.num_heads[i]
        cfg.window_size, cfg.c_e, cfg.c_n = module.window_size, module.out_chans_adj, module.out_chans_node
        cfg.self_condition = int(module.self_condition)
        handle = C.c_void_p()
        native.check(self.lib.dsg_model_create(C.byref(cfg), C.byref(handle)), "dsg_model_create")
        self.handle = handle
        with torch.cuda.device(device):
            self.arena = torch.empty(self.lib.dsg_model_arena_bytes(handle) + 256, dtype=torch.uint8, device=device)
            off = (-self.arena.data_ptr()) % 256
            native.check(self.lib.dsg_model_bind_arena(handle, self.arena.data_ptr() + off,
                                                       self.arena.numel() - off), "dsg_model_bind_arena")
        self.versions = None
        self.workspace = None
        self.ws_key = None

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.dsg_model_destroy(self.handle)
        except Exception:  # interpreter shutdown
            pass

    def keys(self):
        if getattr(self, "_keys", None) is not None:
            return self._keys
        out = []
        key, numel, dtype = C.c_char_p(), C.c_int64(), C.c_int32()
        for i in range(self.lib.dsg_model_num_tensors(self.handle)):
            native.check(self.lib.dsg_model_tensor_info(self.handle, i, C.byref(key), C.byref(numel), C.byref(dtype)),
                         "dsg_model_tensor_info")
            out.append((key.value.decode(), numel.value, dtype.value))
        self._keys = out
        return out

    def differs(self, state) -> bool:
        """Deep staleness probe: does any tensor of `state` differ from the master copy in the arena?"""
        if self.versions is None:
            return True
        st = native.stream_ptr(self.device)
        with torch.cuda.device(self.device):
            flag = torch.zeros(1, dtype=torch.int32, device=self.device)
            keep = []
            for key, numel, dtype in self.keys():
                t = state[key].detach()
                want = torch.int64 if dtype == 1 else torch.float32
                if t.numel() != numel:
                    return True
                if t.device != self.device or t.dtype != want or not t.is_contiguous():
                    t = t.to(device=self.device, dtype=want).contiguous()
                    keep.append(t)
                native.check(self.lib.dsg_model_tensor_differs(self.handle, key.encode(), t.data_ptr(),
                                                               t.numel() * t.element_size(), flag.data_ptr(), st),
                             "dsg_model_tensor_differs")
            return bool(flag.item())

    def upload(self, state):
        with native.device_guard(self.device):
            self._upload(state)

    def _upload(self, state):
        st = native.stream_ptr(self.device)
        keep = []
        for key, numel, dtype in self.keys():
            t = state[key].detach()
            want = torch.int64 if dtype == 1 else torch.float32
            if t.numel() != numel:
                raise native.NativeError(f"{key}: {t.numel()} elements, native model expects {numel}")
            t = t.to(device=self.device, dtype=want).contiguous()
            keep.append(t)
            native.check(self.lib.dsg_model_set_tensor(self.handle, key.encode(), t.data_ptr(),
                                                       t.numel() * t.element_size(), 0, st), "dsg_model_set_tensor")
        native.check(self.lib.dsg_model_finalize(self.handle, st), "dsg_model_finalize")
        del keep  # stream-ordered: the caching allocator keeps the blocks alive until the copies ran

    def skip_info(self):
        stages, granule = C.c_int32(), C.c_int32()
        native.check(self.lib.dsg_model_skip_info(self.handle, C.byref(stages), C.byref(granule)), "dsg_model_skip_info")
        return stages.value, granule.value

    def skip_info2(self):
        granule2 = C.c_int32()
        native.check(self.lib.dsg_model_skip_info2(self.handle, C.byref(granule2)), "dsg_model_skip_info2")
        return granule2.value

    def forward(self, mode, batch, n_cond, adj, node, flags, noise, stride, sc_adj, sc_node, out_adj, out_node,
                skip=None):
        key = (batch, n_cond)
        if self.ws_key != key:
            need = self.lib.dsg_workspace_bytes(self.handle, batch, n_cond)
            self.workspace = None
            with torch.cuda.device(self.device):
                self.workspace = torch.empty(need + 256, dtype=torch.uint8, device=self.device)
            self.ws_key = key
        off = (-self.workspace.data_ptr()) % 256
        a = native.DsgForwardArgs()
        a.struct_size = C.sizeof(native.DsgForwardArgs)
        a.batch, a.n_cond, a.mode = batch, n_cond, mode
        a.adj, a.node, a.flags, a.noise = adj.data_ptr(), node.data_ptr(), flags.data_ptr(), noise.data_ptr()
        a.noise_stride = stride
        a.sc_adj, a.sc_node = native.ptr(sc_adj), native.ptr(sc_node)
        a.out_adj, a.out_node = out_adj.data_ptr(), out_node.data_ptr()
        a.workspace = self.workspace.data_ptr() + off
        a.workspace_bytes = self.workspace.numel() - off
        if skip is not None:
            a.skip_tables, a.skip_table_images, a.skip_buckets = skip.tables.data_ptr(), skip.n_images_cap, len(skip.counts)
            for k, (cnt, side) in enumerate(zip(skip.counts, skip.sides)):
                a.skip_count[k], a.skip_side[k] = cnt, side
            a.skip_phantom_tok0 = skip.phantom_tok0
            base = skip.tables.data_ptr()
            mo = skip.map_offsets
            if "dense_from_c1" in mo:
                a.skip_map_dense_from_c1 = base + 4 * mo["dense_from_c1"]
            else:
                a.skip2_map_c2_from_c1 = base + 4 * mo["c2_from_c1"]
                a.skip2_map_dense_from_c2 = base + 4 * mo["dense_from_c2"]
                a.skip2_map_c2_from_dense = base + 4 * mo["c2_from_dense"]
            if skip.level2 is not None:
                off2, counts2, sides2, phantom2, _ = skip.level2
                a.skip2_tables = skip.tables.data_ptr() + 4 * off2
                a.skip2_table_images, a.skip2_buckets = skip.n_images_cap, len(counts2)
                for k, (cnt, side) in enumerate(zip(counts2, sides2)):
                    a.skip2_count[k], a.skip2_side[k] = cnt, side
                a.skip2_phantom_tok0 = phantom2
        with native.device_guard(self.device):
            native.check(self.lib.dsg_denoiser_forward(self.handle, C.byref(a), native.stream_ptr(self.device)),
                         "dsg_denoiser_forward")

    def debug_buffer(self, name: str, dtype: torch.dtype) -> torch.Tensor:
        """Test hook: flat view of a named activation buffer of the last forward's workspace."""
        off, nbytes = C.c_size_t(), C.c_size_t()
        batch, n_cond = self.ws_key
        native.check(self.lib.dsg_debug_buffer(self.handle, batch, n_cond, name.encode(), C.byref(off), C.byref(nbytes)),
                     "dsg_debug_buffer")
        base = (-self.workspace.data_ptr()) % 256
        return self.workspace[base + off.value: base + off.value + nbytes.value].view(dtype)
