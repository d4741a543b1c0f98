"""Training pass of the native denoiser (SURVEY 8 f-2): forward with saved activations, backward, on native kernels.

What the reference gets from torch autograd when the trainer calls ``loss.backward()``
(runner/trainer/trainer_node_adj.py:171-173) through ``NodeAdjPrecond.forward`` -> ``DiffuseSG.forward``
(model/precond/precond.py:100-105, model/diffusesg/diffusesg.py:765-830) is restated here as ONE autograd node
(`DenoiserTrainFn`) whose forward records a tape of backward closures; every arithmetic step of both directions is a
kernel of libdsg_b200 (tcgen05 GEMMs for every large nn.Linear incl. dgrad and split-K wgrad, row kernels and the
tensor-core attention backward of csrc/backward.cu).  torch supplies device memory, the stream and the autograd hook only.

Parameters live in ONE flat fp32 buffer (`TrainState.flat`; ``nn.Parameter.data`` are views into it, gradients are views
into `TrainState.grad`), so that the optimiser step, the EMA updates and the DDP all-reduce are single launches /
collectives over contiguous memory, and the FiLM generators of all blocks form one matrix.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, List, Optional

import torch
from torch.autograd.function import once_differentiable

from ... import native
from .geometry import block_table, relative_position_index

F32, BF16 = torch.float32, torch.bfloat16
HEAD_DIM = 32
_BIG_SUFFIXES = (".attn.qkv", ".attn.proj", ".mlp.fc1", ".mlp.fc2", ".downsample.reduction", ".upsample.pre_linear",
                 ".upsample.post_linear")


class _PrepJob(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("dst_t", C.c_void_p), ("rows", C.c_int32), ("cols", C.c_int32),
                ("ldd", C.c_int32), ("rows_t", C.c_int32), ("scale_elems", C.c_int64), ("scale", C.c_float),
                ("dst_f32", C.c_int32)]


_FN: Dict[str, object] = {}


def _nc(name: str, *args) -> None:
    fn = _FN.get(name)
    if fn is None:
        fn = _FN[name] = getattr(native.lib(), name)
    rc = fn(*args)
    if rc != 0:
        native.check(rc, name)


def _up(n: int, m: int) -> int:
    return (n + m - 1) // m * m


def _w16_refusal(prefix: str, index: torch.Tensor, shift: int, flags: int) -> Optional[str]:
    """Why the 16 x 16 attention backward (dsg_tr_window_attention_bwd_w16) cannot train this block, or None.  The kernel
    looks the bias up by token offset and rebuilds the SW-MSA mask, so it needs the reference's two buffers (what every
    checkpoint of the reference holds).  Synchronises: call once per block, outside any graph capture."""
    if not torch.equal(index, relative_position_index(16).to(index.device)):
        return (f"training a 16 x 16-window block needs the reference's {prefix}.attn.relative_position_index "
                "(geometry.relative_position_index(16)); this buffer differs")
    if shift > 0 and not flags & native.ATTN_MASK_CANONICAL:
        return (f"training a shifted 16 x 16-window block needs the reference's {prefix}.attn_mask "
                "(geometry.shifted_window_mask); this buffer differs")
    return None


class TrainState:
    """Flat fp32 parameters / gradients and the bf16 GEMM shadows of one DiffuseSG module on one device."""

    def __init__(self, module, device: torch.device):
        assert C.sizeof(_PrepJob) == native.lib().dsg_tr_prep_job_bytes()
        self.module, self.dev = module, device
        self.blocks = block_table(module.img_size, module.embed_dim, module.depths, module.num_heads, module.window_size)
        named = dict(module.named_parameters())
        film_names = ["patch_embed.affine"] + [b["prefix"] + ".affine" for b in self.blocks]
        self.film_off: Dict[str, int] = {}
        off = 0
        for n in film_names:
            self.film_off[n] = off
            off += named[n + ".weight"].shape[0]
        self.film_total = off
        first = [n + ".weight" for n in film_names] + [n + ".bias" for n in film_names]
        first += ["map_layer0.weight", "map_layer0.bias", "map_layer1.weight", "map_layer1.bias"]
        order = first + [k for k in named if k not in set(first)]
        self.offs: Dict[str, int] = {}
        pos = 0
        for k in order:
            self.offs[k] = pos
            pos += _up(named[k].numel(), 4)
        self.numel = pos
        self.order = order
        with native.device_guard(device):
            self.flat = torch.zeros(pos, dtype=F32, device=device)
            self.grad = torch.zeros(pos, dtype=F32, device=device)
        self.shapes = {k: tuple(named[k].shape) for k in order}
        self._wviews: Dict[str, torch.Tensor] = {}
        self.attn_flags: Dict[tuple, int] = {}
        self.w16_refusal: Dict[tuple, Optional[str]] = {}   # 16 x 16 blocks whose buffers the backward kernel cannot take
        for k in order:
            p = named[k]
            view = self.flat[self.offs[k]: self.offs[k] + p.numel()].view(p.shape)
            view.copy_(p.data)
            p.data = view
        self.gviews = {k: self.grad[self.offs[k]: self.offs[k] + named[k].numel()].view(self.shapes[k]) for k in order}
        self.params = named
        self._build_shadows()
        self.anchor = torch.zeros(1, device=device, requires_grad=True)
        self.ddp_group = None      # set by NativeDDP: gradients are all-reduced (mean) over this group during backward
        self.ddp_work: List = []

    # ---- views ---------------------------------------------------------------------------------------------------
    def w(self, key: str) -> torch.Tensor:
        v = self._wviews.get(key)
        if v is None:
            v = self._wviews[key] = self.flat[self.offs[key]: self.offs[key] + math.prod(self.shapes[key])].view(self.shapes[key])
        return v

    def g(self, key: str) -> torch.Tensor:
        return self.gviews[key]

    def attached(self) -> bool:
        """Are the module's parameters still the views into the flat buffer (``.to()`` / a new module would break it)?"""
        base = self.flat.data_ptr()
        return all(self.params[k].data.data_ptr() == base + 4 * self.offs[k] for k in self.order)

    def attach_grads(self) -> bool:
        """Point every ``.grad`` at its view of the flat gradient buffer; returns True when the buffer had to be zeroed
        (some ``.grad`` was None: a fresh step after ``zero_grad(set_to_none=True)``, trainer_node_adj.py:109)."""
        fresh = any(self.params[k].grad is None or self.params[k].grad.data_ptr() != self.gviews[k].data_ptr()
                    for k in self.order)
        if fresh:
            self.grad.zero_()
            for k in self.order:
                self.params[k].grad = self.gviews[k]
        return fresh

    # ---- bf16 shadows --------------------------------------------------------------------------------------------
    def _build_shadows(self):
        m = self.module
        jobs = []
        self.wb: Dict[str, torch.Tensor] = {}    # [N_out, K_in(padded)] bf16: forward operand (and dgrad operand of ConvT)
        self.wbt: Dict[str, torch.Tensor] = {}   # [K_in(padded), N_out] bf16: dgrad operand
        self.qkv_bias: Dict[str, torch.Tensor] = {}
        big = [k[:-7] for k in self.order if k.endswith(".weight") and k[:-7].endswith(_BIG_SUFFIXES)]
        big += ["read_out.0", "read_out.1", "read_out.2", "readout_adj_mlp.fc1", "patch_embed.proj"]
        total = total_t = 0
        plan = []
        for name in big:
            shape = self.shapes[name + ".weight"]
            rows, cols = shape[0], math.prod(shape[1:])
            ldd = 96 if name == "patch_embed.proj" else cols
            plan.append((name, rows, cols, ldd, total, total_t))
            total += _up(rows * ldd, 64)
            total_t += _up(rows * ldd, 64)
        with native.device_guard(self.dev):
            self._wb_flat = torch.zeros(total, dtype=BF16, device=self.dev)
            self._wbt_flat = torch.zeros(max(total_t, 64), dtype=BF16, device=self.dev)
        scale = HEAD_DIM ** -0.5
        for name, rows, cols, ldd, o, ot in plan:
            self.wb[name] = self._wb_flat[o: o + rows * ldd].view(rows, ldd)
            self.wbt[name] = self._wbt_flat[ot: ot + rows * ldd].view(ldd, rows)
            j = _PrepJob()
            j.src, j.dst, j.dst_t = self.w(name + ".weight").data_ptr(), self.wb[name].data_ptr(), self.wbt[name].data_ptr()
            j.rows, j.cols, j.ldd, j.rows_t = rows, cols, ldd, ldd
            j.scale, j.scale_elems, j.dst_f32 = 1.0, 0, 0
            if name.endswith(".attn.qkv"):
                dim = cols
                j.scale, j.scale_elems = scale, dim * dim   # the q rows carry head_dim^-1/2 (diffusesg.py:118)
                with native.device_guard(self.dev):
                    self.qkv_bias[name] = torch.zeros(3 * dim, dtype=F32, device=self.dev)
                jb = _PrepJob()
                jb.src, jb.dst = self.w(name + ".bias").data_ptr(), self.qkv_bias[name].data_ptr()
                jb.rows, jb.cols, jb.ldd, jb.rows_t = 1, 3 * dim, 3 * dim, 3 * dim
                jb.scale, jb.scale_elems, jb.dst_f32 = scale, dim, 1
                jobs.append(jb)
            jobs.append(j)
        arr = (_PrepJob * len(jobs))(*jobs)
        raw = bytes(memoryview(arr).cast("B"))
        self._jobs = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(self.dev)
        self._n_jobs = len(jobs)
        self.shadow_version = None

    def refresh_shadows(self):
        """bf16 copies of the current masters: one launch (call once per forward; the optimiser changes the masters)."""
        _nc("dsg_tr_prep_weights", self._jobs.data_ptr(), self._n_jobs, native.stream_ptr(self.dev))


# ---------------------------------------------------------------------------------------------------------------------
# thin kernel wrappers
# ---------------------------------------------------------------------------------------------------------------------
class _Ops:
    def __init__(self, dev):
        self.dev = dev
        # the stream current when the pass was created (one lookup, not one per launch); None on a CPU device, where only
        # the host-side logic (flat layout, gradient ranges) can run
        self.st = native.stream_ptr(dev) if dev.type == "cuda" else None

    def empty(self, shape, dtype=F32):
        return torch.empty(shape, dtype=dtype, device=self.dev)

    def zeros(self, shape, dtype=F32):
        t = torch.empty(shape, dtype=dtype, device=self.dev)
        t.zero_()   # cudaMemsetAsync
        return t

    def gemm(self, a, w, bias, epi, res=None, out=None):
        """epilogue(a [M, K] @ w [N, K]^T + bias) on the tcgen05 kernel; a, w bf16."""
        m, k = a.shape
        n = w.shape[0]
        if out is None:
            out = self.empty((m, n), BF16 if epi in (native.EPI_BF16, native.EPI_GELU_BF16) else F32)
        _nc("dsg_gemm_bf16", a.data_ptr(), w.data_ptr(), native.ptr(bias), native.ptr(res), out.data_ptr(), m, n, k, epi,
            self.st)
        return out

    def wgrad_mn(self, dy16, x16, dw, scale_rows=0, scale=1.0):
        """dw [N_out, K_in] += dy16 [M, N_out]^T @ x16 [M, x_cols]; both operands bf16 row-major, no transposes."""
        m, n_out = dy16.shape
        x_cols = x16.shape[1]
        out_cols = dw.shape[1]
        bn = 192 if x_cols % 192 == 0 else 128
        tiles = ((n_out + 127) // 128) * ((x_cols + bn - 1) // bn)
        num_kb = (m + 63) // 64
        ksplit = max(1, min(296 // tiles, num_kb // 4))
        _nc("dsg_tr_wgrad", dy16.data_ptr(), x16.data_ptr(), dw.data_ptr(), m, n_out, x_cols, out_cols, ksplit, scale_rows,
            float(scale), self.st)

    def cast_colsum(self, src, colsum=None, cast=False, scale_cols=0, scale=1.0):
        """colsum [C] += column sums of src [M, C] (columns < scale_cols scaled); returns the bf16 copy when asked."""
        m, c = src.shape
        cst = self.empty((m, c), BF16) if cast else None
        if cst is not None or colsum is not None:
            _nc("dsg_tr_cast_colsum", src.data_ptr(), int(src.dtype == BF16), native.ptr(cst), native.ptr(colsum), m, c,
                scale_cols, float(scale), self.st)
        return cst

    def ln_fwd(self, x, gamma, beta, bf16=True, f32=False):
        m, c = x.shape
        y16 = self.empty((m, c), BF16) if bf16 else None
        y32 = self.empty((m, c), F32) if f32 else None
        _nc("dsg_tr_ln_fwd", x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), native.ptr(y16), native.ptr(y32), m, c, self.st)
        return y16, y32

    def ln_bwd(self, dy, x, gamma, dgamma, dbeta, dx_add=None):
        """dx (written over dx_add when given, else a new tensor)."""
        m, c = x.shape
        dx = dx_add if dx_add is not None else self.empty((m, c))
        _nc("dsg_tr_ln_bwd", dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), native.ptr(dx_add), dx.data_ptr(),
            dgamma.data_ptr(), dbeta.data_ptr(), m, c, self.st)
        return dx

    def film_fwd(self, v, film, off, b, l, c):
        out = self.empty(v.shape)
        _nc("dsg_tr_film_silu_fwd", v.data_ptr(), film.data_ptr(), film.shape[1], off, out.data_ptr(), b, l, c, self.st)
        return out

    def film_bwd(self, dout, v, film, off, dfilm, b, l, c):
        dv = self.empty(v.shape)
        _nc("dsg_tr_film_silu_bwd", dout.data_ptr(), v.data_ptr(), film.data_ptr(), film.shape[1], off, dv.data_ptr(),
            dfilm.data_ptr(), b, l, c, self.st)
        return dv

    def gelu(self, pre, dh=None):
        out = self.empty(pre.shape, BF16)
        _nc("dsg_tr_gelu", pre.data_ptr(), native.ptr(dh), out.data_ptr(), pre.numel(), self.st)
        return out

    def gelu_f32(self, pre, dout=None):
        out = self.empty(pre.shape)
        _nc("dsg_tr_gelu_f32", pre.data_ptr(), native.ptr(dout), out.data_ptr(), pre.numel(), self.st)
        return out

    def silu(self, pre, dout=None):
        out = self.empty(pre.shape)
        _nc("dsg_tr_silu", pre.data_ptr(), native.ptr(dout), out.data_ptr(), pre.numel(), self.st)
        return out

    def add_(self, y, x):
        _nc("dsg_tr_add_inplace", y.data_ptr(), x.data_ptr(), y.numel(), self.st)

    def shuffle(self, src, b, h, w, c, to_coarse):
        """fine [b, 2h, 2w, c] <-> coarse [b, h, w, 4, c]"""
        dst = self.empty((b * h * w, 4 * c) if to_coarse else (b * 4 * h * w, c))
        _nc("dsg_tr_shuffle2x2", src.data_ptr(), dst.data_ptr(), b, h, w, c, int(to_coarse), self.st)
        return dst

    def copy_cols(self, src, scol, dst, dcol, ncols, accumulate=False):
        _nc("dsg_tr_copy_cols", src.data_ptr(), src.shape[1], scol, dst.data_ptr(), dst.shape[1], dcol, ncols, src.shape[0],
            int(dst.dtype == BF16), int(accumulate), self.st)

    def sgemm(self, a, a_strides, b, b_strides, m, n, k, bias=None, out=None, accumulate=False, ksplit=1):
        """out [m, n] (+)= sum_k a[m * a_strides[0] + k * a_strides[1]] * b[k * b_strides[0] + n * b_strides[1]]"""
        if out is None:
            ctas = ((m + 63) // 64) * ((n + 63) // 64)
            if ksplit == 1 and ctas < 148 and k >= 2048:      # few output tiles, long contraction: slices meet by atomicAdd
                ksplit = max(1, min(k // 512, 296 // ctas))
            out = self.zeros((m, n)) if ksplit > 1 else self.empty((m, n))
        _nc("dsg_tr_sgemm", a.data_ptr(), int(a.dtype == BF16), a_strides[0], a_strides[1], b.data_ptr(), int(b.dtype == BF16),
            b_strides[0], b_strides[1], native.ptr(bias), out.data_ptr(), out.shape[-1], m, n, k, ksplit,
            int(accumulate or ksplit > 1), self.st)
        return out

    def linear_small(self, x, w, bias):
        """x [M, K] @ w [N, K]^T + bias on the fp32 CUDA-core kernel (fp32 masters, no shadow)."""
        m, k = x.shape
        return self.sgemm(x, (k, 1), w, (1, k), m, w.shape[0], k, bias=bias)

    def linear_small_bwd(self, dy, x, w, dw, db, need_dx=True):
        """dw += dy^T x (dw None: skipped); db += colsum(dy); returns dx = dy w.  dy [M, N] fp32, x [M, K] fp32 / bf16,
        w [N, K]."""
        m, n = dy.shape
        k = x.shape[1]
        if db is not None:
            _nc("dsg_tr_colsum", dy.data_ptr(), db.data_ptr(), m, n, self.st)
        if dw is not None:
            self.sgemm(dy, (1, n), x, (k, 1), n, k, m, out=dw, accumulate=True, ksplit=max(1, min(128, m // 512)))
        if not need_dx:
            return None
        return self.sgemm(dy, (n, 1), w, (k, 1), m, k, n)


# ---------------------------------------------------------------------------------------------------------------------
# the tape
# ---------------------------------------------------------------------------------------------------------------------
class TrainPass:
    """One forward of the denoiser with everything the backward needs; `backward(d_adj, d_node)` fills TrainState.grad
    and, when asked, returns the gradients w.r.t. the input graphs.

    ``params=False`` is the input-only pass (eval mode, or no trainable parameter): its backward runs the data-gradient
    chain alone - no weight-gradient GEMM, no bias column sum, no noise-embedding backward, no all-reduce - and writes
    nothing to TrainState.grad.  The per-channel sums that the LayerNorm and attention backward kernels always accumulate
    land in a scratch buffer instead (`acc`)."""

    def __init__(self, state: TrainState, params: bool = True):
        self.s = state
        self.o = _Ops(state.dev)
        self.params = params
        self.record = True     # False: a no-grad pass - nothing of the forward is kept, GELU rides in the fc1 epilogue
        self._sink = None

    def acc(self, key):
        """Where the backward accumulates the gradient of parameter `key`: its view of TrainState.grad, or in an
        input-only pass a scratch buffer nothing reads (so the sinks of one launch may overlap)."""
        if self.params:
            return self.s.g(key)
        n = math.prod(self.s.shapes[key])
        if self._sink is None or self._sink.numel() < n:
            self._sink = self.o.empty(max(n, 4096))
        return self._sink[:n].view(self.s.shapes[key])

    # -- large linears ---------------------------------------------------------------------------------------------
    def _lin_bwd(self, name, dy, x16, need_dx=True, dx_epi=native.EPI_F32, bias=True, scale_cols=0, transposed_weight=False):
        """Gradients of y = x W^T + b into the flat buffer; returns dx.  dy fp32 or bf16 [M, N_out], x16 bf16 [M, K_in]."""
        s, o = self.s, self.o
        if not self.params:
            if not need_dx:
                return None
            dy16 = dy if dy.dtype == BF16 else o.cast_colsum(dy, cast=True)
            return o.gemm(dy16, s.wb[name] if transposed_weight else s.wbt[name], None, dx_epi)
        db = s.g(name + ".bias") if bias else None
        dw = s.g(name + ".weight")
        dw2 = dw.view(dw.shape[0], -1)
        scale = HEAD_DIM ** -0.5
        dy16 = o.cast_colsum(dy, colsum=db, cast=dy.dtype != BF16, scale_cols=scale_cols, scale=scale)
        if dy.dtype == BF16:
            dy16 = dy
        if transposed_weight:   # ConvTranspose2d weight [in, out]: y = x W, so dW = x^T dy
            o.wgrad_mn(x16, dy16, dw2)
        elif (dw2.shape[1] * 4) % 16 != 0:
            # a weight row that is no multiple of 16 bytes (the 26 / 54-channel embeddings) cannot be a TMA destination:
            # accumulate a zero-padded copy and add its leading columns
            pad = o.zeros((dw2.shape[0], x16.shape[1]))
            o.wgrad_mn(dy16, x16, pad)
            o.copy_cols(pad, 0, dw2, 0, dw2.shape[1], accumulate=True)
        else:
            o.wgrad_mn(dy16, x16, dw2, scale_rows=scale_cols, scale=scale)
        if not need_dx:
            return None
        wd = s.wb[name] if transposed_weight else s.wbt[name]   # [K_in, N_out]
        return o.gemm(dy16, wd, None, dx_epi)

    # -- Swin block ------------------------------------------------------------------------------------------------
    def _block(self, blk, x, film, dfilm, batch):
        s, o, mod = self.s, self.o, self.s.module
        p, dim, res, heads, w, shift = blk["prefix"], blk["dim"], blk["res"], blk["heads"], blk["window"], blk["shift"]
        L = res * res
        foff = s.film_off[p + ".affine"]
        T = w * w
        xf = o.film_fwd(x, film, foff, batch, L, dim)
        y1, _ = o.ln_fwd(xf, s.w(p + ".norm1.weight"), s.w(p + ".norm1.bias"))
        qkv = o.gemm(y1, s.wb[p + ".attn.qkv"], s.qkv_bias[p + ".attn.qkv"], native.EPI_BF16)
        tree = mod.get_submodule(p)
        index = tree.attn.relative_position_index
        mask = tree.attn_mask if shift > 0 else None
        bias = o.empty((heads, T, T))
        _nc("dsg_tr_bias_gather", s.w(p + ".attn.relative_position_bias_table").data_ptr(), index.data_ptr(), bias.data_ptr(),
            heads, T, 0, None, o.st)
        # the mask / bias buffer checks synchronise the stream: once per block (first pass), their result is kept
        fl = s.attn_flags.get((p, batch))
        if fl is None:
            got = C.c_int(0)
            _nc("dsg_window_attention_check", bias.data_ptr(), native.ptr(mask), batch, res, w, shift, heads, o.st, C.byref(got))
            fl = s.attn_flags[(p, batch)] = got.value
            if w == 16:
                s.w16_refusal[(p, batch)] = _w16_refusal(p, index, shift, fl)
        att = o.empty((qkv.shape[0], dim), BF16)
        _nc("dsg_window_attention_flags", qkv.data_ptr(), bias.data_ptr(), native.ptr(mask), att.data_ptr(), batch, res, w, shift,
            heads, fl, o.st)
        xm = o.gemm(att, s.wb[p + ".attn.proj"], s.w(p + ".attn.proj.bias"), native.EPI_RES_F32, res=xf, out=o.empty(xf.shape))
        y2, _ = o.ln_fwd(xm, s.w(p + ".norm2.weight"), s.w(p + ".norm2.bias"))
        if self.record:
            hp = o.gemm(y2, s.wb[p + ".mlp.fc1"], s.w(p + ".mlp.fc1.bias"), native.EPI_BF16)   # pre-activation kept for GELU'
            h = o.gelu(hp)
        else:
            hp, h = None, o.gemm(y2, s.wb[p + ".mlp.fc1"], s.w(p + ".mlp.fc1.bias"), native.EPI_GELU_BF16)
        xo = o.gemm(h, s.wb[p + ".mlp.fc2"], s.w(p + ".mlp.fc2.bias"), native.EPI_RES_F32, res=xm, out=o.empty(xm.shape))

        def bwd(dxo):
            if w == 16 and s.w16_refusal[(p, batch)] is not None:
                raise NotImplementedError(s.w16_refusal[(p, batch)])
            dh = self._lin_bwd(p + ".mlp.fc2", dxo, h, dx_epi=native.EPI_BF16)
            dhp = o.gelu(hp, dh)
            del dh
            dy2 = self._lin_bwd(p + ".mlp.fc1", dhp, y2)
            del dhp
            dxm = o.ln_bwd(dy2, xm, s.w(p + ".norm2.weight"), self.acc(p + ".norm2.weight"), self.acc(p + ".norm2.bias"),
                           dx_add=dxo)
            del dy2
            datt = self._lin_bwd(p + ".attn.proj", dxm, att, dx_epi=native.EPI_BF16)
            dqkv = o.empty(qkv.shape, BF16)
            if w == 16:   # reads the bias table and accumulates its gradient directly (no [heads, T, T] buffer)
                _nc("dsg_tr_window_attention_bwd_w16", qkv.data_ptr(), datt.data_ptr(),
                    s.w(p + ".attn.relative_position_bias_table").data_ptr(), dqkv.data_ptr(),
                    self.acc(p + ".attn.relative_position_bias_table").data_ptr(), batch, res, w, shift, heads, o.st)
            else:
                dbias = o.zeros((heads, T, T))
                _nc("dsg_tr_window_attention_bwd", qkv.data_ptr(), datt.data_ptr(), bias.data_ptr(), native.ptr(mask),
                    dqkv.data_ptr(), dbias.data_ptr(), batch, res, w, shift, heads, o.st)
                if self.params:
                    _nc("dsg_tr_bias_gather", None, index.data_ptr(), dbias.data_ptr(), heads, T, 1,
                        s.g(p + ".attn.relative_position_bias_table").data_ptr(), o.st)
            del datt
            dy1 = self._lin_bwd(p + ".attn.qkv", dqkv, y1, scale_cols=dim)
            del dqkv
            dxf = o.ln_bwd(dy1, xf, s.w(p + ".norm1.weight"), self.acc(p + ".norm1.weight"), self.acc(p + ".norm1.bias"),
                           dx_add=dxm)
            return o.film_bwd(dxf, x, film, foff, dfilm, batch, L, dim)

        return xo, bwd

    def _merge(self, prefix, x, batch, res, dim):
        s, o = self.s, self.o
        g = o.shuffle(x, batch, res // 2, res // 2, dim, True)
        y, _ = o.ln_fwd(g, s.w(prefix + ".norm.weight"), s.w(prefix + ".norm.bias"))
        out = o.gemm(y, s.wb[prefix + ".reduction"], None, native.EPI_F32)

        def bwd(dout):
            dy = self._lin_bwd(prefix + ".reduction", dout, y, bias=False)
            dg = o.ln_bwd(dy, g, s.w(prefix + ".norm.weight"), self.acc(prefix + ".norm.weight"), self.acc(prefix + ".norm.bias"))
            return o.shuffle(dg, batch, res // 2, res // 2, dim, False)

        return out, bwd

    def _breakup(self, prefix, x, skip, batch, res):
        """x, skip [batch * res^2, D / 2] -> [batch * 4 res^2, D / 4]"""
        s, o = self.s, self.o
        c1, c2 = x.shape[1], skip.shape[1]
        d = c1 + c2
        m = x.shape[0]
        xcat = o.empty((m, d), BF16)
        o.copy_cols(x, 0, xcat, 0, c1)
        o.copy_cols(skip, 0, xcat, c1, c2)
        t = o.gemm(xcat, s.wb[prefix + ".pre_linear"], None, native.EPI_F32)
        _, u = o.ln_fwd(t, s.w(prefix + ".norm.weight"), s.w(prefix + ".norm.bias"), bf16=False, f32=True)
        f = o.shuffle(u, batch, res, res, d // 4, False)
        del u
        y, _ = o.ln_fwd(f, s.w(prefix + ".post_norm.weight"), s.w(prefix + ".post_norm.bias"))
        out = o.gemm(y, s.wb[prefix + ".post_linear"], None, native.EPI_F32)

        def bwd(dout):
            dy = self._lin_bwd(prefix + ".post_linear", dout, y, bias=False)
            df = o.ln_bwd(dy, f, s.w(prefix + ".post_norm.weight"), self.acc(prefix + ".post_norm.weight"),
                          self.acc(prefix + ".post_norm.bias"))
            du = o.shuffle(df, batch, res, res, d // 4, True)
            dt = o.ln_bwd(du, t, s.w(prefix + ".norm.weight"), self.acc(prefix + ".norm.weight"), self.acc(prefix + ".norm.bias"))
            dxcat = self._lin_bwd(prefix + ".pre_linear", dt, xcat, bias=False)
            dx, dskip = o.empty((m, c1)), o.empty((m, c2))
            o.copy_cols(dxcat, 0, dx, 0, c1)
            o.copy_cols(dxcat, c1, dskip, 0, c2)
            return dx, dskip

        return out, bwd

    # -- whole network -----------------------------------------------------------------------------------------------
    def forward(self, mode, adj, node, flags, noise, sc_adj, sc_node):
        """mode 0: raw F (noise = c_noise labels); mode 1: EDM-preconditioned D (noise = sigmas).  Returns (adj, node)."""
        s, o, mod = self.s, self.o, self.s.module
        B, ce, n, _ = adj.shape
        cn = node.shape[-1]
        E = mod.embed_dim
        nl = mod.num_layers
        s.refresh_shadows()
        if mode == 1:
            coef = o.empty((4, B))
            _nc("dsg_tr_precond_coef", noise.data_ptr(), coef.data_ptr(), B, o.st)
            c_skip, c_out, c_in, labels = coef[0], coef[1], coef[2], coef[3]
        else:
            c_skip = c_out = c_in = None
            labels = noise
        # noise embedding and the FiLM parameters of every block (:768-771, :236-237)
        pe = o.empty((B, E))
        _nc("dsg_tr_posemb", labels.data_ptr(), pe.data_ptr(), B, E, o.st)
        e0p = o.linear_small(pe, s.w("map_layer0.weight"), s.w("map_layer0.bias"))
        e0 = o.silu(e0p)
        e1p = o.linear_small(e0, s.w("map_layer1.weight"), s.w("map_layer1.bias"))
        emb = o.silu(e1p)
        FT = s.film_total
        wfilm = s.flat[: FT * 512].view(FT, 512)
        bfilm = s.flat[FT * 512: FT * 512 + FT]
        film = o.linear_small(emb, wfilm, bfilm)
        dfilm = o.zeros((B, FT))
        # patch embedding (:562-577)
        M = B * n * n
        inp = o.empty((M, 96), BF16)
        _nc("dsg_tr_embed_input", adj.data_ptr(), node.data_ptr(), native.ptr(sc_adj), native.ptr(sc_node), flags.data_ptr(),
            native.ptr(c_in), inp.data_ptr(), B, n, ce, cn, int(mod.self_condition), 96, o.st)
        t0 = o.gemm(inp, s.wb["patch_embed.proj"], s.w("patch_embed.proj.bias"), native.EPI_F32)
        _, v0 = o.ln_fwd(t0, s.w("patch_embed.norm.weight"), s.w("patch_embed.norm.bias"), bf16=False, f32=True)
        x = o.film_fwd(v0, film, s.film_off["patch_embed.affine"], B, n * n, E)

        def embed_bwd(dx, d_adj, d_node, need_dx):
            dv = o.film_bwd(dx, v0, film, s.film_off["patch_embed.affine"], dfilm, B, n * n, E)
            dt = o.ln_bwd(dv, t0, s.w("patch_embed.norm.weight"), self.acc("patch_embed.norm.weight"),
                          self.acc("patch_embed.norm.bias"))
            dinp = self._lin_bwd("patch_embed.proj", dt, inp, need_dx=need_dx)   # [M, 96] fp32: gradient of the operand
            if not need_dx:
                return None
            del dt
            g_adj, g_node = o.empty(adj.shape), o.empty(node.shape)
            _nc("dsg_tr_embed_input_bwd", dinp.data_ptr(), d_adj.data_ptr(), d_node.data_ptr(), flags.data_ptr(),
                native.ptr(c_in), native.ptr(c_skip), g_adj.data_ptr(), g_node.data_ptr(), B, n, ce, cn,
                int(mod.self_condition), 96, o.st)
            return g_adj, g_node

        # U-Net (:739-756).  seq entries: ("block" | "merge", bwd), ("mark", stage): the output of encoder stage `stage`
        # (its second consumer is the skip concat), ("breakup", bwd, stage whose output is the skip it consumes)
        it = iter(s.blocks)
        seq = []
        skip_x = []
        for st in range(nl):
            dim, res = E << st, n >> st
            for _ in range(mod.depths[st]):
                x, bw = self._block(next(it), x, film, dfilm, B)
                seq.append(("block", bw))
            if st < nl - 1:
                x, bw = self._merge(f"down_layers.{st}.downsample", x, B, res, dim)
                seq.append(("merge", bw))
            skip_x.append(x)
            seq.append(("mark", st))
        for u in range(nl):
            st = nl - 1 - u
            skip = skip_x.pop()              # u == 0: the bottleneck's own output, dropped (:755)
            if u > 0:
                x, bw = self._breakup(f"up_layers.{u}.upsample", x, skip, B, n >> (st + 1))
                seq.append(("breakup", bw, st))
            for _ in range(mod.depths[st]):
                x, bw = self._block(next(it), x, film, dfilm, B)
                seq.append(("block", bw))
        del skip, skip_x
        # heads (:758-825)
        yf, _ = o.ln_fwd(x, s.w("norm.weight"), s.w("norm.bias"))
        r0 = o.gemm(yf, s.wbt["read_out.0"], s.w("read_out.0.bias"), native.EPI_BF16)
        r1 = o.gemm(r0, s.wb["read_out.1"], s.w("read_out.1.bias"), native.EPI_BF16)
        rep = o.gemm(r1, s.wb["read_out.2"], s.w("read_out.2.bias"), native.EPI_F32)
        rep16 = o.cast_colsum(rep, cast=True)
        hap = o.gemm(rep16, s.wb["readout_adj_mlp.fc1"], s.w("readout_adj_mlp.fc1.bias"), native.EPI_BF16)
        ha = o.gelu(hap)
        wa2 = s.w("readout_adj_mlp.fc2.weight")
        narrow = ce <= 8 and E <= 128     # the dedicated warp-per-pixel kernels; otherwise the generic fp32 GEMM
        if narrow:
            tok_a = o.empty((M, ce))
            _nc("dsg_tr_adj_fc2", ha.data_ptr(), wa2.data_ptr(), s.w("readout_adj_mlp.fc2.bias").data_ptr(), tok_a.data_ptr(),
                None, None, M, E, ce, o.st)
        else:
            tok_a = o.sgemm(ha, (E, 1), wa2, (1, E), M, ce, E, bias=s.w("readout_adj_mlp.fc2.bias"))
        out_adj = o.empty(adj.shape)
        _nc("dsg_tr_adj_out", tok_a.data_ptr(), flags.data_ptr(), native.ptr(adj) if mode == 1 else None, native.ptr(c_skip),
            native.ptr(c_out), out_adj.data_ptr(), B, n, ce, 0, o.st)
        pooled = o.empty((B * n, E))
        _nc("dsg_tr_node_pool", rep.data_ptr(), flags.data_ptr(), pooled.data_ptr(), None, None, B, n, E, o.st)
        hnp = o.linear_small(pooled, s.w("readout_node_mlp.fc1.weight"), s.w("readout_node_mlp.fc1.bias"))
        hn = o.gelu_f32(hnp)
        tok_n = o.linear_small(hn, s.w("readout_node_mlp.fc2.weight"), s.w("readout_node_mlp.fc2.bias"))
        out_node = o.empty(node.shape)
        _nc("dsg_tr_node_out", tok_n.data_ptr(), flags.data_ptr(), native.ptr(node) if mode == 1 else None, native.ptr(c_skip),
            native.ptr(c_out), out_node.data_ptr(), B, n, cn, 0, o.st)
        del tok_a, tok_n
        x_final = x

        def heads_bwd(d_adj, d_node):
            dtok_a = o.empty((M, ce))
            _nc("dsg_tr_adj_out", d_adj.data_ptr(), flags.data_ptr(), None, None, native.ptr(c_out), dtok_a.data_ptr(), B, n,
                ce, 1, o.st)
            if narrow:
                if self.params:
                    _nc("dsg_tr_colsum", dtok_a.data_ptr(), s.g("readout_adj_mlp.fc2.bias").data_ptr(), M, ce, o.st)
                    _nc("dsg_tr_adj_fc2", ha.data_ptr(), None, None, None, dtok_a.data_ptr(),
                        s.g("readout_adj_mlp.fc2.weight").data_ptr(), M, E, ce, o.st)
                dha32 = o.sgemm(dtok_a, (ce, 1), wa2, (E, 1), M, E, ce)
            else:
                dha32 = o.linear_small_bwd(dtok_a, ha, wa2, *self._small_grads("readout_adj_mlp.fc2"))
            dha = o.empty((M, E), BF16)
            o.copy_cols(dha32, 0, dha, 0, E)
            del dha32
            dhap = o.gelu(hap, dha)
            del dha
            drep = self._lin_bwd("readout_adj_mlp.fc1", dhap, rep16)
            dtok_n = o.empty((B * n, cn))
            _nc("dsg_tr_node_out", d_node.data_ptr(), flags.data_ptr(), None, None, native.ptr(c_out), dtok_n.data_ptr(), B, n,
                cn, 1, o.st)
            dhn = o.linear_small_bwd(dtok_n, hn, s.w("readout_node_mlp.fc2.weight"), *self._small_grads("readout_node_mlp.fc2"))
            dhnp = o.gelu_f32(hnp, dhn)
            dpooled = o.linear_small_bwd(dhnp, pooled, s.w("readout_node_mlp.fc1.weight"),
                                         *self._small_grads("readout_node_mlp.fc1"))
            _nc("dsg_tr_node_pool", None, flags.data_ptr(), None, dpooled.data_ptr(), drep.data_ptr(), B, n, E, o.st)
            dr1 = self._lin_bwd("read_out.2", drep, r1, dx_epi=native.EPI_BF16)
            dr0 = self._lin_bwd("read_out.1", dr1, r0, dx_epi=native.EPI_BF16)
            dyf = self._lin_bwd("read_out.0", dr0, yf, transposed_weight=True)
            return o.ln_bwd(dyf, x_final, s.w("norm.weight"), self.acc("norm.weight"), self.acc("norm.bias"))

        def cond_bwd():
            demb = o.linear_small_bwd(dfilm, emb, wfilm, s.grad[: FT * 512].view(FT, 512), s.grad[FT * 512: FT * 512 + FT])
            de1p = o.silu(e1p, demb)
            de0 = o.linear_small_bwd(de1p, e0, s.w("map_layer1.weight"), s.g("map_layer1.weight"), s.g("map_layer1.bias"))
            de0p = o.silu(e0p, de0)
            o.linear_small_bwd(de0p, pe, s.w("map_layer0.weight"), s.g("map_layer0.weight"), s.g("map_layer0.bias"),
                               need_dx=False)

        self._seq, self._heads_bwd, self._embed_bwd, self._cond_bwd = seq, heads_bwd, embed_bwd, cond_bwd
        self._nl = nl
        return out_adj, out_node

    def _small_grads(self, name):
        """(dw, db) of a small fp32 layer for linear_small_bwd; (None, None) in an input-only pass."""
        if not self.params:
            return None, None
        return self.s.g(name + ".weight"), self.s.g(name + ".bias")

    def backward(self, d_adj, d_node, need_input=False):
        """Run the tape in reverse; parameter gradients accumulate into TrainState.grad (params=True).  Returns the
        gradients w.r.t. the input graphs (adj, node) when `need_input`, else None."""
        o = self.o
        dx = self._heads_bwd(d_adj, d_node)
        self._heads_bwd = None
        if self.params:
            self._reduce_range("heads")
        seq = self._seq
        pending: Dict[int, torch.Tensor] = {}   # encoder stage -> gradient arriving over its skip connection
        for i in range(len(seq) - 1, -1, -1):
            e = seq[i]
            seq[i] = None
            if e[0] == "mark":
                extra = pending.pop(e[1], None)
                if extra is not None:
                    o.add_(dx, extra)
            elif e[0] == "breakup":
                dx, pending[e[2]] = e[1](dx)
            else:
                dx = e[1](dx)
        out = self._embed_bwd(dx, d_adj, d_node, need_input)
        del dx
        if self.params:
            self._cond_bwd()
            self._reduce_range("rest")
        return out

    def _reduce_range(self, what):
        """DDP: average the gradients over the process group (NCCL all-reduce over NVLink).  The read-out heads' range
        is reduced while the U-Net backward runs; everything else once the tape is done."""
        s = self.s
        if s.ddp_group is None:
            return
        import torch.distributed as dist
        lo = s.offs["read_out.0.weight"]   # flat order: FiLM + noise MLP, embedding, encoder, decoder, then the heads
        rng = s.grad[lo:] if what == "heads" else s.grad[:lo]
        if dist.get_backend(s.ddp_group) == "nccl":
            s.ddp_work.append(dist.all_reduce(rng, op=dist.ReduceOp.AVG, group=s.ddp_group, async_op=True))
        else:   # gloo (the CPU tests of the host logic) has no AVG
            dist.all_reduce(rng, op=dist.ReduceOp.SUM, group=s.ddp_group)
            rng.div_(dist.get_world_size(s.ddp_group))
        if what == "rest":
            for wk in s.ddp_work:
                wk.wait()
            s.ddp_work.clear()


_NO_INPUT_GRAD = {6: "sigmas / noise_labels", 7: "self_cond_x / self_cond_adjs", 8: "self_cond_feat / self_cond_nodes"}


class DenoiserTrainFn(torch.autograd.Function):
    """The whole preconditioned denoiser as one autograd node.  The parameters receive their gradients through ``.grad``
    views of the flat buffer, written by the tape - not through autograd's AccumulateGrad, so the node takes a dummy
    differentiable input that keeps it on the graph.  The input graphs (adj, node) get theirs through autograd when they
    require it (guidance, sensitivity analysis); the noise levels and the self-conditioning inputs have none built."""

    @staticmethod
    def forward(ctx, anchor, tp: TrainPass, mode, adj, node, flags, noise, sc_adj, sc_node):
        out = tp.forward(mode, adj, node, flags, noise, sc_adj, sc_node)
        ctx.tp = tp
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, d_adj, d_node):
        for i, name in _NO_INPUT_GRAD.items():
            if ctx.needs_input_grad[i]:
                raise NotImplementedError(f"DiffuseSG (B200): the gradient w.r.t. {name} is not built (only the input "
                                          "graphs adj / node and the parameters have one); detach that input")
        tp = ctx.tp
        if tp is None:
            raise RuntimeError("DiffuseSG (B200): the training tape is consumed by its first backward (the saved activations "
                               "are released as it runs); backward(retain_graph=True) twice is not supported")
        ctx.tp = None
        s = tp.s
        if tp.params:
            s.attach_grads()
        want_adj, want_node = ctx.needs_input_grad[3], ctx.needs_input_grad[4]
        with native.device_guard(s.dev):
            g = tp.backward(native.require_cuda(d_adj, "grad"), native.require_cuda(d_node, "grad"), want_adj or want_node)
        g_adj, g_node = g if g is not None else (None, None)
        return (None, None, None, g_adj if want_adj else None, g_node if want_node else None, None, None, None, None)


def train_state(module, device) -> TrainState:
    st = module.__dict__.get("_train_state")
    if st is None or st.dev != device or not st.attached():
        st = TrainState(module, device)
        module.__dict__["_train_state"] = st
        module.invalidate_native()
    return st


def run_training_forward(module, mode, adj, node, flags, noise, sc_adj, sc_node, params=True):
    """`DiffuseSG._run` under autograd: returns outputs attached to the autograd graph.  params=False: an input-only tape
    (eval mode or frozen parameters) whose backward gives the input gradients and leaves every parameter gradient alone."""
    dev = adj.device
    st = train_state(module, dev)
    with native.device_guard(dev):
        if not torch.is_grad_enabled():
            # the self-conditioning refresh of a training step (model/precond/precond.py:90-98): same kernels, no tape kept -
            # the fused inference schedule would need its packed weight arena rebuilt after every optimiser step
            tp = TrainPass(st)
            tp.record = False
            out = tp.forward(mode, adj, node, flags, noise, sc_adj, sc_node)
            del tp
            return out
        return DenoiserTrainFn.apply(st.anchor, TrainPass(st, params), mode, adj, node, flags, noise, sc_adj, sc_node)
