"""ctypes binding of libdsg_b200.so (the C ABI declared in include/dsg_b200.h).

There is no fallback: if the shared library is missing or a call fails, a ``NativeError`` is raised.  PyTorch is
used only as the owner of device memory and streams; every pointer crossing the ABI is a raw device pointer.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import functools
import os
from typing import Optional

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libdsg_b200.so")
ABI_VERSION = 4

EPI_BF16, EPI_GELU_BF16, EPI_RES_F32, EPI_F32 = 0, 1, 2, 3
ATTN_MASK_CANONICAL = 1   # dsg_window_attention_check: the mask is the reference's SW-MSA mask


class NativeError(RuntimeError):
    pass


class DsgConfig(C.Structure):
    _fields_ = [("img_size", C.c_int32), ("embed_dim", C.c_int32), ("num_stages", C.c_int32),
                ("depths", C.c_int32 * 4), ("num_heads", C.c_int32 * 4), ("window_size", C.c_int32),
                ("c_e", C.c_int32), ("c_n", C.c_int32), ("self_condition", C.c_int32)]


class DsgForwardArgs(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("batch", C.c_int32), ("n_cond", C.c_int32), ("mode", C.c_int32),
                ("adj", C.c_void_p), ("node", C.c_void_p), ("flags", C.c_void_p), ("noise", C.c_void_p),
                ("noise_stride", C.c_int64), ("sc_adj", C.c_void_p), ("sc_node", C.c_void_p),
                ("out_adj", C.c_void_p), ("out_node", C.c_void_p), ("workspace", C.c_void_p),
                ("workspace_bytes", C.c_size_t), ("skip_tables", C.c_void_p), ("skip_table_images", C.c_int32),
                ("skip_buckets", C.c_int32), ("skip_count", C.c_int32 * 8), ("skip_side", C.c_int32 * 8),
                ("skip_phantom_tok0", C.c_int64), ("skip_map_dense_from_c1", C.c_void_p),
                ("skip2_map_c2_from_c1", C.c_void_p), ("skip2_map_dense_from_c2", C.c_void_p),
                ("skip2_map_c2_from_dense", C.c_void_p), ("skip2_tables", C.c_void_p), ("skip2_table_images", C.c_int32),
                ("skip2_buckets", C.c_int32), ("skip2_count", C.c_int32 * 8), ("skip2_side", C.c_int32 * 8),
                ("skip2_phantom_tok0", C.c_int64)]


class DsgEdmStepParams(C.Structure):
    """include/dsg_b200.h: dsg_edm_step_params (48 bytes; one row per sampler step for CUDA-graph replays)."""
    _fields_ = [("noise_coef", C.c_float), ("inv_t_hat", C.c_float), ("h", C.c_float), ("inv_t_prime", C.c_float),
                ("t_hat", C.c_float), ("reserved", C.c_float), ("seed", C.c_uint64), ("offset_adj", C.c_uint64),
                ("offset_node", C.c_uint64)]


STEP_PARAMS_BYTES = 48
STEP_PARAMS_T_HAT_OFFSET = 16


class DsgProfileClass(C.Structure):
    _fields_ = [("name", C.c_char * 24), ("launches", C.c_uint64), ("ms", C.c_double), ("flops", C.c_double),
                ("bytes", C.c_double)]


_SIGNATURES = {
    "dsg_abi_version": (C.c_int, []),
    "dsg_last_error": (C.c_char_p, []),
    "dsg_launch_count": (C.c_uint64, []),
    "dsg_launch_count_add": (None, [C.c_uint64]),
    "dsg_model_create": (C.c_int, [C.POINTER(DsgConfig), C.POINTER(C.c_void_p)]),
    "dsg_model_destroy": (None, [C.c_void_p]),
    "dsg_model_arena_bytes": (C.c_size_t, [C.c_void_p]),
    "dsg_model_bind_arena": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "dsg_model_num_tensors": (C.c_int, [C.c_void_p]),
    "dsg_model_tensor_info": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_int64),
                                        C.POINTER(C.c_int32)]),
    "dsg_model_set_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "dsg_model_finalize": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dsg_model_tensor_differs": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "dsg_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int, C.c_int]),
    "dsg_model_skip_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dsg_model_skip_info2": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "dsg_denoiser_forward": (C.c_int, [C.c_void_p, C.POINTER(DsgForwardArgs), C.c_void_p]),
    "dsg_edm_pre_step": (C.c_int, [C.c_void_p] * 5 + [C.c_float, C.c_void_p, C.c_void_p] + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_pre_step_philox": (C.c_int, [C.c_void_p] * 3 + [C.c_float, C.c_uint64, C.c_uint64, C.c_int, C.c_uint64, C.c_int,
                                           C.c_void_p, C.c_void_p] + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_post_step": (C.c_int, [C.c_void_p] * 7 + [C.c_float] * 3 + [C.c_void_p] * 2 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_step_advance": (C.c_int, [C.c_void_p] * 4),
    "dsg_edm_pre_step_philox_dev": (C.c_int, [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 4
                                    + [C.c_void_p]),
    "dsg_edm_post_step_dev": (C.c_int, [C.c_void_p] * 10 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_final_step_decode": (C.c_int, [C.c_void_p] * 5 + [C.c_float, C.c_float] + [C.c_void_p] * 6 + [C.c_int] * 6
                                  + [C.c_void_p]),
    "dsg_edm_pre_step_known": (C.c_int, [C.c_void_p] * 7 + [C.c_float] * 2 + [C.c_void_p] * 2 + [C.c_int] * 4
                               + [C.c_void_p]),
    "dsg_edm_pre_step_philox_known": (C.c_int, [C.c_void_p] * 5 + [C.c_float] * 2 + [C.c_uint64, C.c_uint64, C.c_int,
                                      C.c_uint64, C.c_int] + [C.c_void_p] * 3 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_apply_known": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_encode_known": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_guidance_residual": (C.c_int, [C.c_void_p] * 7 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_guidance_update": (C.c_int, [C.c_void_p] * 5 + [C.c_float] + [C.c_void_p] * 2 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_mask_scale": (C.c_int, [C.c_void_p] * 3 + [C.c_float, C.c_void_p, C.c_void_p] + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_decode_samples": (C.c_int, [C.c_void_p] * 6 + [C.c_int] * 6 + [C.c_void_p]),
    "dsg_train_noise": (C.c_int, [C.c_void_p] * 10 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_loss_sums": (C.c_int, [C.c_void_p] * 8 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_edm_loss_sums_backward": (C.c_int, [C.c_void_p] * 10 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_gemm_bf16": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_window_attention": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 5 + [C.c_void_p]),
    "dsg_window_attention_check": (C.c_int, [C.c_void_p] * 2 + [C.c_int] * 5 + [C.c_void_p, C.POINTER(C.c_int)]),
    "dsg_window_attention_flags": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 6 + [C.c_void_p]),
    # training step (SURVEY 8 f-2)
    "dsg_tr_ln_fwd": (C.c_int, [C.c_void_p] * 5 + [C.c_longlong, C.c_int, C.c_void_p]),
    "dsg_tr_ln_bwd": (C.c_int, [C.c_void_p] * 7 + [C.c_longlong, C.c_int, C.c_void_p]),
    "dsg_tr_film_silu_fwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p] + [C.c_int] * 3 + [C.c_void_p]),
    "dsg_tr_film_silu_bwd": (C.c_int, [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 3
                             + [C.c_void_p]),
    "dsg_tr_gelu": (C.c_int, [C.c_void_p] * 3 + [C.c_longlong, C.c_void_p]),
    "dsg_tr_silu": (C.c_int, [C.c_void_p] * 3 + [C.c_longlong, C.c_void_p]),
    "dsg_tr_add_inplace": (C.c_int, [C.c_void_p] * 2 + [C.c_longlong, C.c_void_p]),
    "dsg_tr_wgrad": (C.c_int, [C.c_void_p] * 3 + [C.c_longlong] + [C.c_int] * 5 + [C.c_float, C.c_void_p]),
    "dsg_tr_cast_colsum": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_float,
                                     C.c_void_p]),
    "dsg_tr_shuffle2x2": (C.c_int, [C.c_void_p] * 2 + [C.c_int] * 5 + [C.c_void_p]),
    "dsg_tr_copy_cols": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong,
                                   C.c_int, C.c_int, C.c_void_p]),
    "dsg_tr_embed_input": (C.c_int, [C.c_void_p] * 7 + [C.c_int] * 6 + [C.c_void_p]),
    "dsg_tr_embed_input_bwd": (C.c_int, [C.c_void_p] * 8 + [C.c_int] * 6 + [C.c_void_p]),
    "dsg_tr_adj_out": (C.c_int, [C.c_void_p] * 6 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_tr_node_out": (C.c_int, [C.c_void_p] * 6 + [C.c_int] * 4 + [C.c_void_p]),
    "dsg_tr_adj_fc2": (C.c_int, [C.c_void_p] * 6 + [C.c_longlong, C.c_int, C.c_int, C.c_void_p]),
    "dsg_tr_node_pool": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 3 + [C.c_void_p]),
    "dsg_tr_posemb": (C.c_int, [C.c_void_p] * 2 + [C.c_int] * 2 + [C.c_void_p]),
    "dsg_tr_bias_gather": (C.c_int, [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_void_p, C.c_void_p]),
    "dsg_tr_sgemm": (C.c_int, [C.c_void_p, C.c_int, C.c_longlong, C.c_longlong, C.c_void_p, C.c_int, C.c_longlong,
                               C.c_longlong, C.c_void_p, C.c_void_p, C.c_longlong] + [C.c_int] * 5 + [C.c_void_p]),
    "dsg_tr_gelu_f32": (C.c_int, [C.c_void_p] * 3 + [C.c_longlong, C.c_void_p]),
    "dsg_tr_colsum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "dsg_tr_precond_coef": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "dsg_tr_window_attention_bwd": (C.c_int, [C.c_void_p] * 6 + [C.c_int] * 5 + [C.c_void_p]),
    "dsg_tr_window_attention_bwd_w16": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 5 + [C.c_void_p]),
    "dsg_tr_sumsq": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]),
    "dsg_tr_adam_ema": (C.c_int, [C.c_void_p] * 4 + [C.c_longlong, C.c_void_p] + [C.c_float] * 5 + [C.c_int, C.c_float,
                                  C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_float), C.c_void_p]),
    "dsg_tr_prep_weights": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "dsg_tr_prep_job_bytes": (C.c_int, []),
    "dsg_profile_begin": (C.c_int, [C.c_int]),
    "dsg_profile_read": (C.c_int, [C.POINTER(DsgProfileClass), C.c_int, C.POINTER(C.c_int)]),
    "dsg_profile_dump": (C.c_int, [C.c_char_p]),
    "dsg_profile_stop": (None, []),
    "dsg_proj_ln": (C.c_int, [C.c_void_p] * 7 + [C.c_int, C.c_int, C.c_void_p]),
    "dsg_debug_set_stop_after": (None, [C.c_int]),
    "dsg_debug_set_smem_poison": (None, [C.c_uint, C.c_int]),
    "dsg_debug_buffer": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_char_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
}

_lib: Optional[C.CDLL] = None


def exported_symbols():
    """Every entry point include/dsg_b200.h declares."""
    return sorted(_SIGNATURES)


def lib() -> C.CDLL:
    """Load the shared library (once).  Never builds, never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(f"{LIB_PATH} is missing: build it with `python -m diffusesg_b200.build_native` "
                              "(there is no CPU / PyTorch fallback for this path)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.dsg_abi_version() != ABI_VERSION:
            raise NativeError(f"libdsg_b200 ABI {handle.dsg_abi_version()} != binding ABI {ABI_VERSION}")
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().dsg_last_error()
        raise NativeError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def launch_count() -> int:
    return int(lib().dsg_launch_count())


def profile_begin(pass_stride: int = 1) -> None:
    check(lib().dsg_profile_begin(pass_stride), "dsg_profile_begin")


def profile_read() -> dict:
    """{class name: dict(launches, ms, flops, bytes)} accumulated since profile_begin (waits for the events)."""
    arr = (DsgProfileClass * 8)()
    n = C.c_int()
    check(lib().dsg_profile_read(arr, 8, C.byref(n)), "dsg_profile_read")
    return {arr[i].name.decode(): dict(launches=int(arr[i].launches), ms=arr[i].ms, flops=arr[i].flops,
                                       bytes=arr[i].bytes) for i in range(n.value)}


def profile_dump(path: str) -> None:
    """Per-launch CSV (launch order) of the records gathered since the last profile_read."""
    check(lib().dsg_profile_dump(path.encode()), "dsg_profile_dump")


def profile_stop() -> None:
    lib().dsg_profile_stop()


def device_guard(device):
    """Make `device` current for the duration of a native call (the library's launches and one-time per-device
    setup use the current device); free when it already is."""
    if isinstance(device, torch.device) and device.type != "cuda":
        return contextlib.nullcontext()
    idx = device.index if isinstance(device, torch.device) else device
    if idx is None or torch.cuda.current_device() == idx:
        return contextlib.nullcontext()
    return torch.cuda.device(idx)


def _on_device_of_first_tensor(fn):
    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        t = next((a for a in args if isinstance(a, torch.Tensor) and a.is_cuda), None)
        if t is None:
            return fn(*args, **kwargs)
        with device_guard(t.device):
            return fn(*args, **kwargs)
    return wrapped


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def require_cuda(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    if not t.is_cuda:
        raise NativeError(f"{name} must live on a CUDA device: the B200 path has no CPU implementation")
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


# ---------------------------------------------------------------------------------------------------------
# thin functional wrappers (used by the kernel-level parity tests)
# ---------------------------------------------------------------------------------------------------------
@_on_device_of_first_tensor
def gemm_bf16(a: torch.Tensor, w: torch.Tensor, bias=None, res=None, epi: int = EPI_F32) -> torch.Tensor:
    """epilogue(a [M,K] @ w [N,K]^T + bias) on the tcgen05 kernel.  a, w: bf16 CUDA."""
    assert a.is_cuda and a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16
    a, w = a.contiguous(), w.contiguous()
    m, k = a.shape
    n = w.shape[0]
    out = torch.empty(m, n, device=a.device, dtype=torch.bfloat16 if epi in (EPI_BF16, EPI_GELU_BF16) else torch.float32)
    check(lib().dsg_gemm_bf16(ptr(a), ptr(w), ptr(bias), ptr(res), ptr(out), m, n, k, epi, stream_ptr(a.device)),
          "dsg_gemm_bf16")
    return out


@_on_device_of_first_tensor
def window_attention(qkv: torch.Tensor, bias: torch.Tensor, mask, batch: int, res: int, window: int, shift: int,
                     heads: int) -> torch.Tensor:
    assert qkv.is_cuda and qkv.dtype == torch.bfloat16
    out = torch.empty(qkv.shape[0], heads * 32, device=qkv.device, dtype=torch.bfloat16)
    check(lib().dsg_window_attention(ptr(qkv.contiguous()), ptr(bias.contiguous()), ptr(mask), ptr(out), batch, res,
                                     window, shift, heads, stream_ptr(qkv.device)), "dsg_window_attention")
    return out


@_on_device_of_first_tensor
def edm_pre_step(adj, node, eps_adj, eps_node, flags, noise_coef: float):
    b, ce, n, _ = adj.shape
    cn = node.shape[-1]
    adj_hat, node_hat = torch.empty_like(adj), torch.empty_like(node)
    check(lib().dsg_edm_pre_step(ptr(adj), ptr(node), ptr(eps_adj), ptr(eps_node), ptr(flags), float(noise_coef),
                                 ptr(adj_hat), ptr(node_hat), b, ce, n, cn, stream_ptr(adj.device)), "dsg_edm_pre_step")
    return adj_hat, node_hat


def _aten_normal_policy(numel: int, dev: torch.device):
    """(grid, counter_offset) ATen uses for `normal_` on a float tensor of `numel` elements
    (ATen/native/cuda/DistributionTemplates.h: calc_execution_policy, block 256, unroll 4)."""
    props = torch.cuda.get_device_properties(dev)
    blocks_per_sm = props.max_threads_per_multi_processor // 256
    grid = min(props.multi_processor_count * blocks_per_sm, (numel + 255) // 256)
    return grid, ((numel - 1) // (256 * grid * 4) + 1) * 4


@_on_device_of_first_tensor
def edm_pre_step_fused_noise(adj, node, flags, noise_coef: float):
    """edm_pre_step with eps_adj = randn_like(adj), eps_node = randn_like(node) drawn inside the kernel from the
    current torch CUDA generator state, which is advanced exactly as the two randn_like calls would advance it
    (bit-identical results, no eps tensors; tests/test_gpu_kernels.py::test_edm_pre_step_fused_noise_matches_torch)."""
    b, ce, n, _ = adj.shape
    cn = node.shape[-1]
    dev = adj.device
    gen = torch.cuda.default_generators[dev.index if dev.index is not None else torch.cuda.current_device()]
    seed, off = gen.initial_seed(), gen.get_offset()
    grid_a, inc_a = _aten_normal_policy(adj.numel(), dev)
    grid_n, inc_n = _aten_normal_policy(node.numel(), dev)
    gen.set_offset(off + inc_a + inc_n)
    adj_hat, node_hat = torch.empty_like(adj), torch.empty_like(node)
    check(lib().dsg_edm_pre_step_philox(ptr(adj), ptr(node), ptr(flags), float(noise_coef), seed, off, grid_a, off + inc_a,
                                        grid_n, ptr(adj_hat), ptr(node_hat), b, ce, n, cn, stream_ptr(dev)),
          "dsg_edm_pre_step_philox")
    return adj_hat, node_hat


@_on_device_of_first_tensor
def edm_pre_step_known(adj, node, eps_adj, eps_node, known, flags, noise_coef: float, t_hat: float):
    """Completion pre-step with caller-drawn noise: mask(isnan(k) ? x + noise_coef * eps : k + t_hat * eps);
    known = (known_adj, known_node), NaN on free entries."""
    b, ce, n, _ = adj.shape
    cn = node.shape[-1]
    adj_hat, node_hat = torch.empty_like(adj), torch.empty_like(node)
    check(lib().dsg_edm_pre_step_known(ptr(adj), ptr(node), ptr(eps_adj), ptr(eps_node), ptr(known[0]), ptr(known[1]),
                                       ptr(flags), float(noise_coef), float(t_hat), ptr(adj_hat), ptr(node_hat), b, ce, n,
                                       cn, stream_ptr(adj.device)), "dsg_edm_pre_step_known")
    return adj_hat, node_hat


@_on_device_of_first_tensor
def edm_pre_step_fused_noise_known(adj, node, known, flags, noise_coef: float, t_hat: float):
    """edm_pre_step_known with eps drawn inside the kernel exactly as edm_pre_step_fused_noise draws it (same values,
    same generator advance)."""
    b, ce, n, _ = adj.shape
    cn = node.shape[-1]
    dev = adj.device
    gen = torch.cuda.default_generators[dev.index if dev.index is not None else torch.cuda.current_device()]
    seed, off = gen.initial_seed(), gen.get_offset()
    grid_a, inc_a = _aten_normal_policy(adj.numel(), dev)
    grid_n, inc_n = _aten_normal_policy(node.numel(), dev)
    gen.set_offset(off + inc_a + inc_n)
    adj_hat, node_hat = torch.empty_like(adj), torch.empty_like(node)
    check(lib().dsg_edm_pre_step_philox_known(ptr(adj), ptr(node), ptr(known[0]), ptr(known[1]), ptr(flags),
                                              float(noise_coef), float(t_hat), seed, off, grid_a, off + inc_a, grid_n, None,
                                              ptr(adj_hat), ptr(node_hat), b, ce, n, cn, stream_ptr(dev)),
          "dsg_edm_pre_step_philox_known")
    return adj_hat, node_hat


@_on_device_of_first_tensor
def edm_apply_known(adj, node, known, flags):
    """In place: x = mask(isnan(k) ? x : k) on both tensors (the completion rule after the last step)."""
    b, ce, n, _ = adj.shape
    cn = node.shape[-1]
    check(lib().dsg_edm_apply_known(ptr(adj), ptr(node), ptr(known[0]), ptr(known[1]), ptr(flags), b, ce, n, cn,
                                    stream_ptr(adj.device)), "dsg_edm_apply_known")
    return adj, node


@_on_device_of_first_tensor
def edm_guidance_residual(d_adj, d_node, known, flags):
    """Output gradient of 1/2 sum_known (D - k)^2: r = mask(isnan(k) ? 0 : D - k) on both tensors (new tensors)."""
    b, ce, n, _ = d_adj.shape
    cn = d_node.shape[-1]
    r_adj, r_node = torch.empty_like(d_adj), torch.empty_like(d_node)
    check(lib().dsg_edm_guidance_residual(ptr(d_adj), ptr(d_node), ptr(known[0]), ptr(known[1]), ptr(flags), ptr(r_adj),
                                          ptr(r_node), b, ce, n, cn, stream_ptr(d_adj.device)), "dsg_edm_guidance_residual")
    return r_adj, r_node


@_on_device_of_first_tensor
def edm_guidance_update(d_adj, d_node, g_adj, g_node, flags, w: float):
    """In place: D = mask(D - w G) on both tensors (the guided denoiser output)."""
    b, ce, n, _ = d_adj.shape
    cn = d_node.shape[-1]
    check(lib().dsg_edm_guidance_update(ptr(d_adj), ptr(d_node), ptr(g_adj), ptr(g_node), ptr(flags), float(w), ptr(d_adj),
                                        ptr(d_node), b, ce, n, cn, stream_ptr(d_adj.device)), "dsg_edm_guidance_update")
    return d_adj, d_node


@_on_device_of_first_tensor
def encode_known(node_cls, bbox, adj_cls, batch: int, c_e: int, n: int, c_n: int, device):
    """(known_adj [B,c_e,N,N], known_node [B,N,c_n]) fp32 from int32 classes (-1 = free) and boxes (NaN = free); any
    input may be None.  Inputs are not validated here (runner/mcmc_sampler/completion.py does that)."""
    known_adj = torch.empty(batch, c_e, n, n, dtype=torch.float32, device=device)
    known_node = torch.empty(batch, n, c_n, dtype=torch.float32, device=device)
    with device_guard(known_adj.device):
        check(lib().dsg_encode_known(ptr(node_cls), ptr(bbox), ptr(adj_cls), ptr(known_adj), ptr(known_node), batch, c_e,
                                     n, c_n, stream_ptr(known_adj.device)), "dsg_encode_known")
    return known_adj, known_node


def aten_normal_policy(numel: int, dev: torch.device):
    return _aten_normal_policy(numel, dev)


_FUSED_NOISE_OK = {}


def fused_noise_ok(dev: torch.device) -> bool:
    """One-time self-check per device: does the in-kernel Philox stream (which restates ATen's private launch policy
    for ``normal_``: block 256, unroll 4, grid cap, counter increment) still reproduce ``torch.randn_like`` x 2 on the
    installed torch, values AND generator advance?  If not (a torch upgrade changed the policy) the sampler keeps the
    two ``randn_like`` launches instead of silently drawing a different stream.  The global generator is left
    untouched."""
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key in _FUSED_NOISE_OK:
        return _FUSED_NOISE_OK[key]
    gen = torch.cuda.default_generators[key]
    saved = gen.get_state()
    try:
        with device_guard(dev):
            adj = torch.zeros(2, 3, 16, 16, device=dev)
            node = torch.zeros(2, 16, 5, device=dev)
            flags = torch.ones(2, 16, dtype=torch.bool, device=dev)
            gen.manual_seed(0x5EED)
            a, n = edm_pre_step_fused_noise(adj, node, flags, 1.0)      # 0 + 1 * eps == eps
            probe = torch.rand(4, device=dev)
            gen.manual_seed(0x5EED)
            ra, rn = torch.randn_like(adj), torch.randn_like(node)
            rprobe = torch.rand(4, device=dev)
            ok = bool(torch.equal(a, ra) and torch.equal(n, rn) and torch.equal(probe, rprobe))
    finally:
        gen.set_state(saved)
    if not ok:
        import warnings
        warnings.warn("diffusesg_b200: the fused Philox noise no longer matches torch.randn_like on this torch build "
                      f"({torch.__version__}); falling back to torch.randn_like launches (and eager steps)")
    _FUSED_NOISE_OK[key] = ok
    return ok


@_on_device_of_first_tensor
def edm_final_step_decode(adj_hat, node_hat, d1, flags, inv_t_hat: float, h: float, num_adj_type: int,
                          num_node_type: int, want_state: bool = True, cur_params: Optional[int] = None):
    """Last (Euler) sampler step fused with the decode of the final sample: returns
    (adj_next | None, node_next | None, adj_cls int32 [B,N,N], node_cls int32 [B,N], bbox fp32 [B,N,4])."""
    b, ce, n, _ = adj_hat.shape
    cn = node_hat.shape[-1]
    dev = adj_hat.device
    adj_next = torch.empty_like(adj_hat) if want_state else None
    node_next = torch.empty_like(node_hat) if want_state else None
    adj_cls = torch.empty(b, n, n, dtype=torch.int32, device=dev)
    node_cls = torch.empty(b, n, dtype=torch.int32, device=dev)
    bbox = torch.empty(b, n, 4, dtype=torch.float32, device=dev)
    check(lib().dsg_edm_final_step_decode(ptr(adj_hat), ptr(node_hat), ptr(d1[0]), ptr(d1[1]), ptr(flags), float(inv_t_hat),
                                          float(h), cur_params, ptr(adj_next), ptr(node_next), ptr(adj_cls), ptr(node_cls),
                                          ptr(bbox), int(num_adj_type), int(num_node_type), b, ce, n, cn, stream_ptr(dev)),
          "dsg_edm_final_step_decode")
    return adj_next, node_next, adj_cls, node_cls, bbox


@_on_device_of_first_tensor
def edm_post_step(adj_hat, node_hat, d1, d2, flags, inv_t_hat: float, h: float, inv_t_prime: float):
    b, ce, n, _ = adj_hat.shape
    cn = node_hat.shape[-1]
    adj_next, node_next = torch.empty_like(adj_hat), torch.empty_like(node_hat)
    d2a, d2n = (None, None) if d2 is None else d2
    check(lib().dsg_edm_post_step(ptr(adj_hat), ptr(node_hat), ptr(d1[0]), ptr(d1[1]), ptr(d2a), ptr(d2n), ptr(flags),
                                  float(inv_t_hat), float(h), float(inv_t_prime), ptr(adj_next), ptr(node_next), b, ce,
                                  n, cn, stream_ptr(adj_hat.device)), "dsg_edm_post_step")
    return adj_next, node_next


@_on_device_of_first_tensor
def edm_mask_scale(adj, node, flags, scale: float):
    b, ce, n, _ = adj.shape
    cn = node.shape[-1]
    adj_out, node_out = torch.empty_like(adj), torch.empty_like(node)
    check(lib().dsg_edm_mask_scale(ptr(adj), ptr(node), ptr(flags), float(scale), ptr(adj_out), ptr(node_out), b, ce, n,
                                   cn, stream_ptr(adj.device)), "dsg_edm_mask_scale")
    return adj_out, node_out


def _flags_u8(flags: torch.Tensor) -> torch.Tensor:
    return (flags if flags.dtype == torch.uint8 else flags.to(torch.uint8)).contiguous()


@_on_device_of_first_tensor
def train_noise(clean_adj, clean_node, eps_adj, eps_node, sigmas, flags):
    """(noisy_adj, noise_adj, noisy_node, noise_node) of the EDM training objective, one fused launch."""
    clean_adj, clean_node = require_cuda(clean_adj, "clean_adj"), require_cuda(clean_node, "clean_node")
    eps_adj, eps_node = require_cuda(eps_adj, "eps_adj"), require_cuda(eps_node, "eps_node")
    sigmas = require_cuda(sigmas, "sigmas")
    b, ce, n, _ = clean_adj.shape
    cn = clean_node.shape[-1]
    f = _flags_u8(flags)
    outs = [torch.empty_like(clean_adj), torch.empty_like(clean_adj), torch.empty_like(clean_node),
            torch.empty_like(clean_node)]
    check(lib().dsg_train_noise(ptr(clean_adj), ptr(clean_node), ptr(eps_adj), ptr(eps_node), ptr(sigmas), ptr(f),
                                ptr(outs[0]), ptr(outs[1]), ptr(outs[2]), ptr(outs[3]), b, ce, n, cn,
                                stream_ptr(clean_adj.device)), "dsg_train_noise")
    return tuple(outs)


@_on_device_of_first_tensor
def edm_loss_sums(pred_adj, target_adj, pred_node, target_node, weights, flags):
    """([B] masked weighted squared-error sum over the adjacency tensor, [B] over the node tensor)."""
    pred_adj, target_adj = require_cuda(pred_adj, "pred_adj"), require_cuda(target_adj, "target_adj")
    pred_node, target_node = require_cuda(pred_node, "pred_node"), require_cuda(target_node, "target_node")
    w = None if weights is None else require_cuda(weights.reshape(-1), "loss_weight")
    b, ce, n, _ = pred_adj.shape
    cn = pred_node.shape[-1]
    f = _flags_u8(flags)
    s_adj = torch.empty(b, device=pred_adj.device, dtype=torch.float32)
    s_node = torch.empty_like(s_adj)
    check(lib().dsg_edm_loss_sums(ptr(pred_adj), ptr(target_adj), ptr(pred_node), ptr(target_node), ptr(w), ptr(f),
                                  ptr(s_adj), ptr(s_node), b, ce, n, cn, stream_ptr(pred_adj.device)),
          "dsg_edm_loss_sums")
    return s_adj, s_node


class _EdmLossSums(torch.autograd.Function):
    """Autograd node around the fused loss reduction: forward dsg_edm_loss_sums, backward dsg_edm_loss_sums_backward."""

    @staticmethod
    def forward(ctx, pred_adj, target_adj, pred_node, target_node, weights, flags):
        s_adj, s_node = edm_loss_sums(pred_adj.detach(), target_adj, pred_node.detach(), target_node, weights, flags)
        ctx.save_for_backward(pred_adj.detach(), target_adj, pred_node.detach(), target_node,
                              weights if weights is not None else torch.empty(0, device=pred_adj.device), flags)
        ctx.has_w = weights is not None
        return s_adj, s_node

    @staticmethod
    def backward(ctx, g_adj, g_node):
        pred_adj, target_adj, pred_node, target_node, w, flags = ctx.saved_tensors
        pa, ta = require_cuda(pred_adj, "pred_adj"), require_cuda(target_adj, "target_adj")
        pn, tn = require_cuda(pred_node, "pred_node"), require_cuda(target_node, "target_node")
        wv = require_cuda(w.reshape(-1), "loss_weight") if ctx.has_w else None
        b, ce, n, _ = pa.shape
        cn = pn.shape[-1]
        f = _flags_u8(flags)
        ga, gn = require_cuda(g_adj.contiguous(), "grad"), require_cuda(g_node.contiguous(), "grad")
        gd_a, gd_n = torch.empty_like(pa), torch.empty_like(pn)
        with device_guard(pa.device):
            check(lib().dsg_edm_loss_sums_backward(ptr(pa), ptr(ta), ptr(pn), ptr(tn), ptr(wv), ptr(f), ptr(ga), ptr(gn),
                                                   ptr(gd_a), ptr(gd_n), b, ce, n, cn, stream_ptr(pa.device)),
                  "dsg_edm_loss_sums_backward")
        return gd_a, None, gd_n, None, None, None


def edm_loss_sums_autograd(pred_adj, target_adj, pred_node, target_node, weights, flags):
    """edm_loss_sums with an autograd graph to the predictions (targets / weights / flags are constants)."""
    return _EdmLossSums.apply(pred_adj, target_adj, pred_node, target_node, weights, flags)


@_on_device_of_first_tensor
def decode_samples(adj, node, flags, num_adj_type: int, num_node_type: int):
    """int32 edge classes [B,N,N], int32 node classes [B,N], fp32 boxes [B,N,4] of a final sample, on the device."""
    b, ce, n, _ = adj.shape
    cn = node.shape[-1]
    adj_cls = torch.empty(b, n, n, dtype=torch.int32, device=adj.device)
    node_cls = torch.empty(b, n, dtype=torch.int32, device=adj.device)
    bbox = torch.empty(b, n, 4, dtype=torch.float32, device=adj.device)
    check(lib().dsg_decode_samples(ptr(adj), ptr(node), ptr(flags), ptr(adj_cls), ptr(node_cls), ptr(bbox),
                                   int(num_adj_type), int(num_node_type), b, ce, n, cn, stream_ptr(adj.device)),
          "dsg_decode_samples")
    return adj_cls, node_cls, bbox
