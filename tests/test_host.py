"""CPU-only checks: the C ABI library loads and exports what include/dsg_b200.h declares, host-side logic of the
drop-in classes, and the world_size-2 sharded sampling path over gloo.  No compute call needs a GPU here."""
import copy
import ctypes as C
import json
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

from diffusesg_b200 import native
from diffusesg_b200.model.diffusesg.diffusesg import DiffuseSG
from diffusesg_b200.model.precond.precond import NodeAdjPrecond
from diffusesg_b200.runner.mcmc_sampler.edm import NodeAdjEDMSampler
from diffusesg_b200.runner.objectives.edm import get_preconditioning_params
from diffusesg_b200.runner.sampler.sharded import per_gpu_batch, shard_bounds
from diffusesg_b200.utils.synthetic import CONFIGS, in_chans, synthetic_inputs, synthetic_state_dict
from oracle import denoiser_oracle as O
from oracle import edm_oracle as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _module(cfg):
    return DiffuseSG(img_size=cfg["img"], in_chans=in_chans(cfg), patch_size=1, embed_dim=cfg["embed"],
                     depths=cfg["depths"], num_heads=[3, 6, 12, 24], window_size=cfg["window"], mlp_ratio=4.,
                     drop_rate=0., attn_drop_rate=0., drop_path_rate=0.0, self_condition=cfg["self_cond"],
                     symmetric_noise=False, out_chans_adj=cfg["c_e"], out_chans_node=cfg["c_n"])


def _native_cfg(cfg):
    c = native.DsgConfig()
    c.img_size, c.embed_dim, c.num_stages = cfg["img"], cfg["embed"], len(cfg["depths"])
    for i, (d, h) in enumerate(zip(cfg["depths"], cfg["heads"])):
        c.depths[i], c.num_heads[i] = d, h
    c.window_size, c.c_e, c.c_n, c.self_condition = cfg["window"], cfg["c_e"], cfg["c_n"], int(cfg["self_cond"])
    return c


# ---------------------------------------------------------------------------------------------------------
# C ABI
# ---------------------------------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "dsg_b200.h")).read()
    declared = sorted(set(re.findall(r"DSG_API[^;]*?\b(dsg_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 20
    lib = native.lib()
    for name in declared:
        assert hasattr(lib, name), f"{name} is declared in include/dsg_b200.h but not exported"
    assert declared == native.exported_symbols()
    assert lib.dsg_abi_version() == native.ABI_VERSION == 4


@pytest.mark.parametrize("name", ["vg", "coco", "tiny", "n64w16"])
def test_native_tensor_table_matches_reference_state_dict(name, golden_dir):
    ref = json.load(open(os.path.join(golden_dir, f"layout_{name}.json")))["layout"]
    lib = native.lib()
    h = C.c_void_p()
    native.check(lib.dsg_model_create(C.byref(_native_cfg(CONFIGS[name])), C.byref(h)), "create")
    try:
        assert lib.dsg_model_num_tensors(h) == len(ref)
        key, numel, dtype = C.c_char_p(), C.c_int64(), C.c_int32()
        for i, (k, shape, dt) in enumerate(ref):
            native.check(lib.dsg_model_tensor_info(h, i, C.byref(key), C.byref(numel), C.byref(dtype)), "info")
            assert key.value.decode() == k
            assert numel.value == int(np.prod(shape))
            assert dtype.value == (1 if dt == "int64" else 0)
        assert lib.dsg_model_arena_bytes(h) > 4 * sum(int(np.prod(s)) for _, s, _ in ref)
        small, big = lib.dsg_workspace_bytes(h, 2, 1), lib.dsg_workspace_bytes(h, 8, 1)
        assert 0 < small < big
    finally:
        lib.dsg_model_destroy(h)


def test_native_error_paths_without_gpu():
    lib = native.lib()
    bad = _native_cfg(CONFIGS["vg"])
    bad.num_heads[0] = 4                                   # 96 channels need 3 heads of 32
    h = C.c_void_p()
    assert lib.dsg_model_create(C.byref(bad), C.byref(h)) == 1
    assert b"heads" in lib.dsg_last_error()
    h = C.c_void_p()
    native.check(lib.dsg_model_create(C.byref(_native_cfg(CONFIGS["tiny"])), C.byref(h)), "create")
    try:
        buf = (C.c_float * 4)()
        assert lib.dsg_model_set_tensor(h, b"norm.weight", buf, 16, 1, None) == 3        # no arena bound
        assert lib.dsg_model_finalize(h, None) == 3
        args = native.DsgForwardArgs()
        args.struct_size = C.sizeof(native.DsgForwardArgs)
        assert lib.dsg_denoiser_forward(h, C.byref(args), None) == 3                     # not finalized
        assert lib.dsg_model_bind_arena(h, C.c_void_p(256), 16) == 5                     # arena too small
    finally:
        lib.dsg_model_destroy(h)


# ---------------------------------------------------------------------------------------------------------
# drop-in module
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["vg", "coco", "tiny", "n64w16"])
def test_module_state_dict_is_the_reference_layout(name, golden_dir):
    ref = json.load(open(os.path.join(golden_dir, f"layout_{name}.json")))
    m = _module(CONFIGS[name])
    sd = m.state_dict()
    assert list(sd) == [k for k, _, _ in ref["layout"]]
    for (k, shape, dt), v in zip(ref["layout"], sd.values()):
        assert list(v.shape) == shape and str(v.dtype) == "torch." + dt, k
    assert sum(p.numel() for p in m.parameters()) == ref["n_params"]
    m.load_state_dict(synthetic_state_dict(CONFIGS[name]), strict=True)
    wrapped = NodeAdjPrecond(precond="edm", model=m, self_condition=True, symmetric_noise=False)
    assert list(wrapped.state_dict()) == ["model." + k for k in sd]


def test_module_buffers_match_reference_init(golden_dir):
    ref = json.load(open(os.path.join(golden_dir, "layout_vg.json")))["init_sums"]
    sd = _module(CONFIGS["vg"]).state_dict()
    for k, v in sd.items():
        if k.endswith("relative_position_index") or k.endswith("attn_mask"):
            assert float(v.double().sum()) == ref[k][0] and float(v.double().abs().sum()) == ref[k][1], k


def test_module_deepcopy_and_unsupported_options():
    m = _module(CONFIGS["tiny"])
    m2 = copy.deepcopy(m)                                  # ema_pytorch.EMA does this (learning_utils.py:160)
    assert m2._nat is None and list(m2.state_dict()) == list(m.state_dict())
    with pytest.raises(NotImplementedError):
        DiffuseSG(img_size=16, in_chans=13, patch_size=4, depths=[1], num_heads=[3], window_size=4, drop_path_rate=0.,
                  symmetric_noise=False, out_chans_adj=3, out_chans_node=5)
    with pytest.raises(NotImplementedError):
        NodeAdjPrecond(precond="vp", model=m, self_condition=True, symmetric_noise=False)


def test_forward_refuses_cpu_tensors():
    cfg = CONFIGS["tiny"]
    m = _module(cfg).eval()
    adj, node, flags, sigmas, _, _ = synthetic_inputs(cfg, 2, seed=7)
    with torch.no_grad(), pytest.raises(native.NativeError):
        m(adj, node, flags, sigmas.log() / 4)


def test_preconditioning_params_match_oracle():
    s = torch.tensor([80.0, 3.0, 0.5, 0.002])
    for a, b in zip(get_preconditioning_params("edm", s), O.precond_coefficients(s)):
        assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------
# sampler host logic
# ---------------------------------------------------------------------------------------------------------
def _sampler(steps=256):
    return NodeAdjEDMSampler(num_steps=steps, clip_samples=True, clip_samples_min=-1.0, clip_samples_max=1.0,
                             clip_samples_scope="x_0", dev="cpu", objective="edm", self_condition=True,
                             symmetric_noise=False)


def test_sampler_schedule_matches_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "sampler_tiny.npz"))
    np.testing.assert_array_equal(_sampler(256).sigma_steps.numpy(), g["sigma_steps_256"])
    s8 = _sampler(8)
    t = torch.cat([s8.sigma_steps, torch.zeros(1, dtype=torch.float64)]).to(torch.float32)
    np.testing.assert_array_equal(t.numpy(), g["t_steps"])


def test_sampler_step_scalars_match_oracle_bit_for_bit():
    s = _sampler(256)
    ts = E.t_steps_fp32(256)
    for i in range(256):
        got, want = s.step_scalars(ts[i], ts[i + 1]), E.step_scalars(ts[i], ts[i + 1], 256)
        assert got["noise_coef"] == float(want["noise_coef"]) and got["h"] == float(want["h"])
        assert got["inv_t_hat"] == float(1.0 / want["t_hat"]) and float(got["t_hat"]) == float(want["t_hat"])
        if i < 255:
            assert got["inv_t_prime"] == float(1.0 / want["t_prime"])
    assert s.step_scalars(ts[0], ts[1])["gamma"] == 0.0          # sigma = 80 is outside [S_min, S_max]
    assert s.step_scalars(ts[100], ts[101])["gamma"] == pytest.approx(40 / 256)


def test_sampler_rejects_unbuilt_variants():
    with pytest.raises(NotImplementedError):
        NodeAdjEDMSampler(num_steps=8, solver="euler", clip_samples=False, clip_samples_min=None, clip_samples_max=None,
                          clip_samples_scope="x_0", dev="cpu", self_condition=True, symmetric_noise=False)
    with pytest.raises(NotImplementedError):
        NodeAdjEDMSampler(num_steps=8, clip_samples=False, clip_samples_min=None, clip_samples_max=None,
                          clip_samples_scope="x_0", dev="cpu", self_condition=True, symmetric_noise=True)


class _Cfg(dict):
    """ml_collections.ConfigDict stand-in: attribute access + `in`."""
    __getattr__ = dict.__getitem__


def test_factories_take_the_reference_config_keys():
    from diffusesg_b200.utils.learning_utils import get_network
    from diffusesg_b200.utils.sampling_utils import get_mc_sampler, load_model
    cfg = _Cfg(dev="cpu", flag_sg=True, logdir="/tmp", dataset=_Cfg(name="visual_genome_sg", max_node_num=64),
               model=_Cfg(name="diffuse_sg", feature_dims=[96], depths=[1, 1, 3, 1], window_size=8, patch_size=1),
               train=_Cfg(self_cond=True, node_encoding="bits", edge_encoding="bits", resume=None),
               mcmc=_Cfg(name="edm", precond="edm", sigma_dist="edm", num_steps=256,
                         sample_clip=_Cfg(min=-1.0, max=1.0, scope="x_0")))
    model = get_network(cfg, None)
    assert isinstance(model, NodeAdjPrecond) and len(model.state_dict()) == 247
    assert sum(p.numel() for p in model.parameters()) == 35813660
    sampler = get_mc_sampler(cfg)
    assert sampler.num_steps == 256 and sampler.S_churn == 40 and sampler.S_noise == 1.003
    ckpt = {"model": {"module." + k: v.clone() for k, v in model.state_dict().items()}}   # DDP-prefixed checkpoint
    load_model(ckpt, model, "model")


# ---------------------------------------------------------------------------------------------------------
# multi-GPU host path: world_size 2 over gloo
# ---------------------------------------------------------------------------------------------------------
def test_shard_bounds_cover_everything():
    for total in (0, 1, 7, 512, 1000):
        for world in (1, 2, 3, 8):
            spans = [shard_bounds(total, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(e - b for b, e in spans) - min(e - b for b, e in spans) <= 1
    assert per_gpu_batch(512, 4) == 128 and per_gpu_batch(2, 8) == 1


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from diffusesg_b200.runner.sampler.sharded import sample_sharded, seed_everything
    from diffusesg_b200.utils.dist_training import gather_tensors
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        seed_everything(1234, rank)
        n, ce, cn = 8, 2, 3
        flags = torch.arange(n)[None, :] < torch.arange(2, 9)[:, None]       # 7 graphs: uneven split 4 + 3

        class FakeSampler:                                                   # stands in for the GPU sampler
            dev = "cpu"

            def sample(self, model, node_flags, num_node_chan, num_edge_chan):
                b = node_flags.shape[0]
                cnt = node_flags.sum(1).float()
                return (cnt.view(b, 1, 1, 1).expand(b, num_edge_chan, n, n).clone(),
                        (cnt * 10 + rank).view(b, 1, 1).expand(b, n, num_node_chan).clone())

        a, nd = sample_sharded(FakeSampler(), None, flags, batch_size=4, num_node_chan=cn, num_edge_chan=ce)
        g = gather_tensors(torch.full((2, 3), float(rank)), 0, "cpu")
        torch.save(dict(a=a, n=nd, g=g, draw=torch.randn(2)), os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_sharded_sampling_world_size_2_gloo(tmp_path):
    import torch.multiprocessing as mp
    port = 29500 + os.getpid() % 2000
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "r0.pt"), torch.load(tmp_path / "r1.pt")
    assert torch.equal(r0["a"], r1["a"]) and torch.equal(r0["n"], r1["n"])       # every rank holds the full result
    assert r0["a"].shape == (7, 2, 8, 8) and r0["n"].shape == (7, 8, 3)
    assert r0["a"][:, 0, 0, 0].tolist() == [2, 3, 4, 5, 6, 7, 8]                 # rank order, padding trimmed
    assert r0["n"][:, 0, 0].tolist() == [20, 30, 40, 50, 61, 71, 81]             # rows 0-3 from rank 0, 4-6 from rank 1
    assert r0["g"][:, 0].tolist() == [0, 0, 1, 1]
    assert not torch.equal(r0["draw"], r1["draw"])                               # seed + rank


def test_aten_normal_policy_matches_calc_execution_policy(monkeypatch):
    """Launch grid and Philox counter increment ATen uses for `normal_` on a float CUDA tensor
    (ATen/native/cuda/DistributionTemplates.h::calc_execution_policy, block 256, unroll 4) - the fused-noise pre-step
    advances the torch generator by exactly this much."""
    import types

    from diffusesg_b200 import native

    props = types.SimpleNamespace(multi_processor_count=148, max_threads_per_multi_processor=2048)
    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda dev: props)
    dev = torch.device("cuda", 0)
    # VG adjacency state at batch 512: 512 * 6 * 64 * 64 elements -> the full grid of 148 * 8 blocks, 11 float4 per thread
    assert native._aten_normal_policy(512 * 6 * 64 * 64, dev) == (1184, 44)
    assert native._aten_normal_policy(512 * 64 * 12, dev) == (1184, 4)
    assert native._aten_normal_policy(1000, dev) == (4, 4)
    assert native._aten_normal_policy(1, dev) == (1, 4)
    assert native._aten_normal_policy(1184 * 256 * 4 + 1, dev) == (1184, 8)



@pytest.mark.parametrize("n,granule,counts", [(64, 16, [2, 9, 16, 17, 33, 48, 62, 5, 64, 1]), (40, 10, [33, 2, 10, 11, 21, 30, 40]),
                                              (16, 4, [1, 4, 5, 8, 14, 3, 16])])
def test_skip_plan_host_tables(n, granule, counts):
    """Host side of the padding skipping (include/dsg_b200.h: dsg_model_skip_info): the compact layout must show every
    sample exactly once, inside a corner that covers its last valid node, bucket by bucket, with even image counts
    (the 8 x 8 attention kernel pairs windows) and one all-padding phantom image in the bucket of side `granule`."""
    import numpy as np
    from diffusesg_b200.model.diffusesg.diffusesg import SkipPlan
    b = len(counts)
    flags = torch.arange(n)[None, :] < torch.tensor(counts)[:, None]
    flags[0, 0] = False                       # holes are allowed: only the LAST valid node matters
    table, cnt, sides, phantom_tok0, pixels = SkipPlan.host_tables(flags, n, granule)
    cap = b + SkipPlan.TABLE_EXTRA
    assert len(table) == SkipPlan.table_len(b)
    perm, tok0, width = table[:sum(cnt)], table[cap:cap + b], table[cap + b:cap + 2 * b]
    assert sorted(p for p in perm if p >= 0) == list(range(b))
    assert sides == sorted(sides) and sides[0] == granule and all(s % granule == 0 and s <= n for s in sides)
    assert all(c % 2 == 0 and c > 0 for c in cnt)
    assert pixels == sum(c * s * s for c, s in zip(cnt, sides))
    img, tok = 0, 0
    phantom_seen = False
    for c, s in zip(cnt, sides):
        for k in range(c):
            p = perm[img + k]
            if p >= 0:
                assert width[p] == s and tok0[p] == tok + k * s * s
                assert s >= counts[p] and (s - granule < counts[p] or s == granule)     # smallest corner that covers it
            elif s == granule and tok + k * s * s == phantom_tok0:
                phantom_seen = True
        img += c
        tok += c * s * s
    assert phantom_seen
    # more than 8 distinct corner sizes cannot be expressed: the caller then keeps the dense schedule
    many = torch.arange(64)[None, :] < torch.arange(1, 65, 7)[:, None]
    assert SkipPlan.host_tables(many, 64, 4) is None


def test_step_params_row_layout():
    """The per-step table the captured graphs read (dsg_edm_step_params, 48 bytes): the numpy packing of graphs.py and
    the ctypes mirror of native.py must agree field by field."""
    import ctypes as C
    import numpy as np
    from diffusesg_b200 import native
    assert C.sizeof(native.DsgEdmStepParams) == native.STEP_PARAMS_BYTES == 48
    assert native.DsgEdmStepParams.t_hat.offset == native.STEP_PARAMS_T_HAT_OFFSET
    dt = np.dtype([("noise_coef", "<f4"), ("inv_t_hat", "<f4"), ("h", "<f4"), ("inv_t_prime", "<f4"), ("t_hat", "<f4"),
                   ("reserved", "<f4"), ("seed", "<u8"), ("offset_adj", "<u8"), ("offset_node", "<u8")])
    assert dt.itemsize == 48
    for name, _ in native.DsgEdmStepParams._fields_:
        assert dt.fields[name][1] == getattr(native.DsgEdmStepParams, name).offset, name


def test_skip_plan_row_maps_compose():
    """The row maps between the dense grid and the two compact layouts (dsg_forward_args.skip_map_* / skip2_map_*): reading
    a tensor through the maps must reproduce it inside every kept corner and deliver the phantom's token outside."""
    import numpy as np
    from diffusesg_b200.model.diffusesg.diffusesg import SkipPlan
    n, g1, g2, stages = 64, 16, 32, 2
    counts = [2, 9, 16, 17, 33, 48, 62, 5, 64, 31]
    b, res = len(counts), n >> stages
    flags = torch.arange(n)[None, :] < torch.tensor(counts)[:, None]
    t1, c1, s1, ph1, _ = SkipPlan.host_tables(flags, n, g1)
    t2, c2, s2, ph2, px2 = SkipPlan.host_tables(flags, n, g2)
    cap = b + SkipPlan.TABLE_EXTRA
    maps = SkipPlan.row_maps(t1, c1, s1, ph1, b, n, stages, (t2, c2, s2, ph2))
    only1 = SkipPlan.row_maps(t1, c1, s1, ph1, b, n, stages)["dense_from_c1"]
    w1, w2 = t1[cap + b:cap + 2 * b] >> stages, t2[cap + b:cap + 2 * b] >> stages
    n1 = sum(c * (s >> stages) ** 2 for c, s in zip(c1, s1))
    n2 = px2 >> (2 * stages)
    assert len(maps["c2_from_c1"]) == len(maps["c2_from_dense"]) == n2 and len(maps["dense_from_c2"]) == b * res * res
    assert maps["c2_from_c1"].max() < n1 and maps["dense_from_c2"].max() < n2 and maps["c2_from_dense"].max() < b * res * res
    # a tensor in the first compact layout: value = 1000 b + 16 r + x inside the corners, -7 at the phantom, -1 elsewhere
    x1 = np.full(n1, -1.0)
    dense_ref = np.full((b, res, res), -7.0)
    for k in range(b):
        idx = SkipPlan.corner_index(t1[cap:cap + b], t1[cap + b:cap + 2 * b], stages, k, res)
        rr, xx = np.nonzero(idx >= 0)
        x1[idx[rr, xx]] = 1000 * k + 16 * rr + xx
        dense_ref[k, rr, xx] = 1000 * k + 16 * rr + xx
    phantom1 = ph1 >> (2 * stages)
    x1[phantom1:phantom1 + (g1 >> stages) ** 2] = -7.0
    assert np.array_equal(x1[only1].reshape(b, res, res), dense_ref)                      # level 1 only: dense <- c1
    x2 = x1[maps["c2_from_c1"]]                                                            # c2 <- c1
    dense = x2[maps["dense_from_c2"]].reshape(b, res, res)                                  # dense <- c2
    for k in range(b):                                                                      # the level-2 corner survives, -7 outside
        assert np.array_equal(dense[k, :w2[k], :w2[k]], dense_ref[k, :w2[k], :w2[k]])
        outside = np.ones((res, res), bool)
        outside[:w2[k], :w2[k]] = False
        assert (dense[k][outside] == -7.0).all()
        assert w1[k] <= w2[k]
    back = dense_ref.reshape(-1)[maps["c2_from_dense"]]                                     # c2 <- dense
    keep = x2 != -7.0
    assert np.array_equal(back[keep], x2[keep])


# ---------------------------------------------------------------------------------------------------------
# training step, host logic (SURVEY 8 f-2): flat parameter layout, ema_pytorch's decay schedule, data-parallel ranges
# ---------------------------------------------------------------------------------------------------------
def test_train_state_flat_layout():
    from diffusesg_b200.model.diffusesg.train_graph import TrainState
    m = _module(CONFIGS["tiny"])
    before = {k: v.detach().clone() for k, v in m.named_parameters()}
    ts = TrainState(m, torch.device("cpu"))
    assert ts.attached() and ts.numel % 4 == 0
    for k, p in m.named_parameters():
        assert torch.equal(p.data, before[k]) and ts.offs[k] % 4 == 0, k               # values kept, 16-byte aligned
        assert p.data.data_ptr() == ts.flat.data_ptr() + 4 * ts.offs[k], k               # views into the flat buffer
    spans = sorted((ts.offs[k], ts.offs[k] + before[k].numel()) for k in before)
    assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:]))                           # no overlap
    # the FiLM generators of all blocks form ONE [film_total, 512] matrix at the start, their biases follow
    ft = ts.film_total
    assert ft == sum(v.shape[0] for k, v in before.items() if k.endswith("affine.weight"))
    w = ts.flat[: ft * 512].view(ft, 512)
    off = ts.film_off["down_layers.1.blocks.1.affine"]
    assert torch.equal(w[off: off + 384], before["down_layers.1.blocks.1.affine.weight"])
    assert torch.equal(ts.flat[ft * 512 + off: ft * 512 + off + 384], before["down_layers.1.blocks.1.affine.bias"])
    # the read-out range (reduced first under DDP) is the tail of the buffer and holds nothing else
    lo = ts.offs["read_out.0.weight"]
    tail = {k for k in before if ts.offs[k] >= lo}
    assert tail == {k for k in before if k.startswith(("read_out.", "norm.", "readout_"))}
    assert ts.attach_grads() and not ts.attach_grads()
    assert all(p.grad.data_ptr() == ts.grad.data_ptr() + 4 * ts.offs[k] for k, p in m.named_parameters())
    m2 = copy.deepcopy(m)                                    # the EMA copy gets its own storage, not the flat views
    assert m2.__dict__.get("_train_state") is None
    assert next(m2.parameters()).data_ptr() != next(m.parameters()).data_ptr()


def test_native_ema_follows_the_ema_pytorch_schedule():
    """ema_pytorch.EMA(beta, update_every=1, update_after_step=0, inv_gamma=1, power=1): copy, copy, then
    decay = min(beta, 1 - 1 / (1 + epoch)), epoch = number of updates so far (utils/learning_utils.py:148-166)."""
    from diffusesg_b200.utils.train_utils import NativeEMA
    e = NativeEMA.__new__(NativeEMA)
    e.beta, e.step, e.initted = 0.9, 0, False
    e.denoiser = types.SimpleNamespace(invalidate_native=lambda: None)
    got = []
    for _ in range(12):
        got.append(e.next_decay())
        e._advance()
    want = [0.0, 0.0] + [min(0.9, 1 - 1 / (1 + k)) for k in range(2, 12)]
    assert got == pytest.approx(want)


def _ddp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from diffusesg_b200.model.diffusesg.train_graph import TrainPass
    from diffusesg_b200.utils.train_utils import NativeDDP, find_denoiser
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        torch.manual_seed(100 + rank)                       # different initial weights per rank
        net = _module(CONFIGS["tiny"])
        with torch.no_grad():
            for p in net.parameters():
                p.add_(torch.randn_like(p) * 0.01)
        model = NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False)
        ddp = NativeDDP(model)
        ts = find_denoiser(ddp).__dict__["_train_state"]
        ts.attach_grads()
        ts.grad.fill_(float(rank + 1))                      # what a backward on this rank would have left
        tp = TrainPass(ts)
        tp._reduce_range("heads")
        lo = ts.offs["read_out.0.weight"]
        mid = (float(ts.grad[:lo].mean()), float(ts.grad[lo:].mean()))
        tp._reduce_range("rest")
        torch.save(dict(flat=ts.flat.clone(), grad=ts.grad.clone(), mid=mid), os.path.join(out_dir, f"d{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_native_ddp_world_size_2_gloo(tmp_path):
    import torch.multiprocessing as mp
    port = 31500 + os.getpid() % 2000
    mp.spawn(_ddp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    d0, d1 = torch.load(tmp_path / "d0.pt"), torch.load(tmp_path / "d1.pt")
    assert torch.equal(d0["flat"], d1["flat"])                                   # parameters broadcast from rank 0
    assert d0["mid"] == (1.0, 1.5) and d1["mid"] == (2.0, 1.5)                   # read-out range reduced first
    assert float(d0["grad"].min()) == 1.5 == float(d0["grad"].max()) and torch.equal(d0["grad"], d1["grad"])


def test_fused_adam_checkpoint_round_trip():
    """optimizer.state_dict() / load_state_dict(): moments stored per parameter name, step count and lr restored."""
    from diffusesg_b200.utils.train_utils import FusedAdam
    m = NodeAdjPrecond(precond="edm", model=_module(CONFIGS["tiny"]), self_condition=True, symmetric_noise=False)
    opt = FusedAdam(m, lr=3e-4, weight_decay=0.01)
    torch.manual_seed(0)
    opt.m.normal_()
    opt.v.uniform_()
    opt.steps = 17
    opt.param_groups[0]["lr"] = 1.5e-4
    sd = opt.state_dict()
    assert set(sd["state"]) == {k for k, _ in m.model.named_parameters()}
    assert sd["state"]["norm.weight"]["exp_avg"].shape == (96,)
    m2 = NodeAdjPrecond(precond="edm", model=_module(CONFIGS["tiny"]), self_condition=True, symmetric_noise=False)
    opt2 = FusedAdam(m2, lr=1.0)
    opt2.load_state_dict(sd)
    assert opt2.steps == 17 and opt2.param_groups[0]["lr"] == 1.5e-4 and opt2.param_groups[0]["weight_decay"] == 0.01
    ts, ts2 = opt.ts, opt2.ts
    for k in ts.order:
        n = ts.params[k].numel()
        assert torch.equal(opt2.m[ts2.offs[k]: ts2.offs[k] + n], opt.m[ts.offs[k]: ts.offs[k] + n]), k
        assert torch.equal(opt2.v[ts2.offs[k]: ts2.offs[k] + n], opt.v[ts.offs[k]: ts.offs[k] + n]), k
    with pytest.raises(ValueError):
        opt2.load_state_dict({"state": {}})


# ---------------------------------------------------------------------------------------------------------
# bench.py --dump-outputs
# ---------------------------------------------------------------------------------------------------------
def test_bench_dump_outputs_whole_batch_or_seeded_subset(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    outs = {"adjs": torch.arange(64.).view(8, 2, 2, 2), "nodes": torch.arange(16.).view(8, 2)}   # 40 bytes per graph
    bench.dump_outputs(str(tmp_path / "all"), outs)
    assert np.array_equal(np.load(tmp_path / "all" / "adjs.npy"), outs["adjs"].numpy())
    assert np.array_equal(np.load(tmp_path / "all" / "nodes.npy"), outs["nodes"].numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 5 * 40 + 39)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), outs)
    a, n = np.load(tmp_path / "s1" / "adjs.npy"), np.load(tmp_path / "s1" / "nodes.npy")
    assert a.dtype == np.float32 and n.dtype == np.float32 and a.shape == (5, 2, 2, 2) and n.shape == (5, 2)
    assert np.array_equal(a[:, 0, 0, 0] / 8, n[:, 0] / 2)          # the same graphs from both arrays
    assert np.array_equal(a, np.load(tmp_path / "s2" / "adjs.npy"))  # and the same ones on every run
