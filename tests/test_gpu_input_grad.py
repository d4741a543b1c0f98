"""Gradients w.r.t. the input graphs through the native denoiser, and guided scene-graph completion, on the B200 (run with
-m gpu): the embedding-input backward kernel against an fp64 torch adjoint, the whole denoiser's input gradients against
torch autograd of the fp32 CPU oracle, the side effects of an input-gradient call, and sample_completion with
reconstruction guidance against the guided completion oracle (DESIGN.md §3.7)."""
import ctypes as C

import numpy as np
import pytest
import torch

from diffusesg_b200 import native
from diffusesg_b200.model.diffusesg.diffusesg import DiffuseSG
from diffusesg_b200.model.precond.precond import NodeAdjPrecond
from diffusesg_b200.runner.mcmc_sampler import completion
from diffusesg_b200.runner.mcmc_sampler.edm import NodeAdjEDMSampler
from diffusesg_b200.utils.synthetic import CONFIGS, in_chans, synthetic_inputs, synthetic_state_dict
from oracle import completion_oracle as CO
from oracle import guided_completion_oracle as GO
from oracle import denoiser_oracle as O

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
NAN = float("nan")
LD = 96


def _rel(a, b):
    return float((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm().clamp_min(1e-30))


# ---------------------------------------------------------------------------------------------------------
# the embedding-input backward kernel
# ---------------------------------------------------------------------------------------------------------
def _embed_input_ref(adj, node, flags, c_in, self_cond, sc_adj, sc_node):
    """embed_input_kernel restated in torch (any dtype): [B n n, LD] with the self-conditioning planes first, the adjacency
    planes unmasked, the node planes of i and of j masked by flag_i flag_j, zero padding."""
    b, ce, n, _ = adj.shape
    ci = c_in.view(-1, 1, 1, 1) if c_in is not None else 1.0
    pair = (flags[:, :, None] & flags[:, None, :]).to(adj.dtype)[..., None]           # [B, n, n, 1]
    a = (ci * adj).permute(0, 2, 3, 1)                                               # [B, n, n, ce]
    cnode = (ci[..., 0] if c_in is not None else 1.0) * node                           # [B, n, cn]
    ni = cnode[:, :, None, :].expand(b, n, n, -1)
    nj = cnode[:, None, :, :].expand(b, n, n, -1)
    if self_cond:
        sa = sc_adj.permute(0, 2, 3, 1)
        si, sj = sc_node[:, :, None, :].expand(b, n, n, -1), sc_node[:, None, :, :].expand(b, n, n, -1)
        parts = [sa, a, si * pair, ni * pair, sj * pair, nj * pair]
    else:
        parts = [a, ni * pair, nj * pair]
    x = torch.cat(parts, -1)
    return torch.nn.functional.pad(x, (0, LD - x.shape[-1])).reshape(b * n * n, LD)


def _adjoint_ref(dinp, g_adj, g_node, flags, c_in, c_skip, self_cond, sc_adj, sc_node, adj, node):
    """fp64 autograd of <dinp, embed_input(adj, node)> + <g_adj, c_skip pair adj> + <g_node, c_skip flag node>."""
    a = adj.double().requires_grad_(True)
    x = node.double().requires_grad_(True)
    ci = None if c_in is None else c_in.double()
    inp = _embed_input_ref(a, x, flags, ci, self_cond, sc_adj.double(), sc_node.double())
    loss = (inp * dinp.double()).sum()
    if c_skip is not None:
        pair = (flags[:, None, :, None] & flags[:, None, None, :]).double()
        loss = loss + (g_adj.double() * c_skip.double().view(-1, 1, 1, 1) * pair * a).sum()
        loss = loss + (g_node.double() * c_skip.double().view(-1, 1, 1) * flags[..., None].double() * x).sum()
    ga, gx = torch.autograd.grad(loss, (a, x))
    return ga, gx


def _launch_embed_bwd(dinp, g_adj, g_node, flags, c_in, c_skip, self_cond, b, n, ce, cn):
    d_adj = torch.empty(b, ce, n, n, device=DEV)
    d_node = torch.empty(b, n, cn, device=DEV)
    native.check(native.lib().dsg_tr_embed_input_bwd(dinp.data_ptr(), native.ptr(g_adj), native.ptr(g_node),
                                                     flags.data_ptr(), native.ptr(c_in), native.ptr(c_skip),
                                                     d_adj.data_ptr(), d_node.data_ptr(), b, n, ce, cn, int(self_cond), LD,
                                                     native.stream_ptr(DEV)), "dsg_tr_embed_input_bwd")
    return d_adj, d_node


def _embed_case(b, n, ce, cn, counts, seed):
    g = torch.Generator().manual_seed(seed)
    flags = torch.arange(n)[None, :] < torch.tensor(counts)[:, None]
    flags[0, 1] = False                   # a hole in the middle of a sample, not only trailing padding
    t = lambda *s: torch.randn(*s, generator=g)
    return dict(dinp=t(b * n * n, LD), g_adj=t(b, ce, n, n), g_node=t(b, n, cn), flags=flags,
                c_in=torch.rand(b, generator=g) + 0.2, c_skip=torch.rand(b, generator=g), adj=t(b, ce, n, n),
                node=t(b, n, cn), sc_adj=t(b, ce, n, n), sc_node=t(b, n, cn))


EMBED_SHAPES = [(3, 16, 3, 5, [16, 9, 3]), (2, 64, 6, 12, [62, 17]), (2, 40, 3, 12, [33, 40]), (2, 20, 4, 6, [20, 7])]


@pytest.mark.parametrize("b,n,ce,cn,counts", EMBED_SHAPES)
@pytest.mark.parametrize("self_cond", [True, False])
@pytest.mark.parametrize("mode", [0, 1])
def test_embed_input_backward_matches_fp64_adjoint(b, n, ce, cn, counts, self_cond, mode):
    c = _embed_case(b, n, ce, cn, counts, seed=b * n + ce)
    c_in, c_skip = (c["c_in"], c["c_skip"]) if mode == 1 else (None, None)
    want_a, want_n = _adjoint_ref(c["dinp"], c["g_adj"], c["g_node"], c["flags"], c_in, c_skip, self_cond, c["sc_adj"],
                                  c["sc_node"], c["adj"], c["node"])
    dv = lambda t: None if t is None else t.to(DEV).contiguous()
    args = (dv(c["dinp"]), dv(c["g_adj"]), dv(c["g_node"]), dv(c["flags"]), dv(c_in), dv(c_skip), self_cond, b, n, ce, cn)
    got_a, got_n = _launch_embed_bwd(*args)
    again_a, again_n = _launch_embed_bwd(*args)
    ea, en = _rel(got_a, want_a), _rel(got_n, want_n)
    assert ea < 1e-5 and en < 1e-5, (ea, en)
    assert torch.equal(got_a, again_a) and torch.equal(got_n, again_n)        # deterministic: no atomics
    pad = ~c["flags"].to(DEV)
    assert float(got_n[pad].abs().sum()) == 0.0


def test_embed_input_backward_ignores_shared_memory_leftovers():
    b, n, ce, cn, counts = EMBED_SHAPES[1]
    c = _embed_case(b, n, ce, cn, counts, seed=3)
    dv = lambda t: t.to(DEV).contiguous()
    args = (dv(c["dinp"]), dv(c["g_adj"]), dv(c["g_node"]), dv(c["flags"]), dv(c["c_in"]), dv(c["c_skip"]), True, b, n, ce,
            cn)
    out = []
    for poison in (0, 1):
        native.lib().dsg_debug_set_smem_poison(0x7fc00000, poison)
        try:
            _launch_embed_bwd(*args)          # leaves the poison behind for the next launch
            out.append(_launch_embed_bwd(*args))
        finally:
            native.lib().dsg_debug_set_smem_poison(0, 0)
    torch.cuda.synchronize()
    assert torch.equal(out[0][0], out[1][0]) and torch.equal(out[0][1], out[1][1])


# ---------------------------------------------------------------------------------------------------------
# the guidance kernels
# ---------------------------------------------------------------------------------------------------------
def test_guidance_kernels_bit_exact():
    g = torch.Generator(device=DEV).manual_seed(4)
    b, ce, n, cn = 3, 4, 16, 7
    flags = (torch.arange(n, device=DEV)[None, :] < torch.tensor([16, 9, 4], device=DEV)[:, None]).contiguous()
    pair = (flags[:, None, :, None] & flags[:, None, None, :])
    rows = flags[..., None]
    d_adj = torch.randn(b, ce, n, n, device=DEV, generator=g) * pair
    d_node = torch.randn(b, n, cn, device=DEV, generator=g) * rows
    ka = torch.where(pair & (torch.rand(b, ce, n, n, device=DEV, generator=g) < 0.5),
                     torch.randn(b, ce, n, n, device=DEV, generator=g), NAN)
    kn = torch.where(rows & (torch.rand(b, n, cn, device=DEV, generator=g) < 0.5),
                     torch.randn(b, n, cn, device=DEV, generator=g), NAN)
    ra, rn = native.edm_guidance_residual(d_adj, d_node, (ka, kn), flags)
    assert torch.equal(ra, torch.where(pair & ~ka.isnan(), d_adj - ka, 0.0))
    assert torch.equal(rn, torch.where(rows & ~kn.isnan(), d_node - kn, 0.0))
    ga, gn = torch.randn(b, ce, n, n, device=DEV, generator=g), torch.randn(b, n, cn, device=DEV, generator=g)
    w = 0.37
    want_a, want_n = torch.where(pair, d_adj - w * ga, 0.0), torch.where(rows, d_node - w * gn, 0.0)
    got_a, got_n = native.edm_guidance_update(d_adj.clone(), d_node.clone(), ga, gn, flags, w)
    assert torch.equal(got_a, want_a) and torch.equal(got_n, want_n)


# ---------------------------------------------------------------------------------------------------------
# the whole denoiser: input gradients against autograd of the CPU oracle
# ---------------------------------------------------------------------------------------------------------
def _net(cfg, sd):
    net = DiffuseSG(img_size=cfg["img"], in_chans=in_chans(cfg), patch_size=1, embed_dim=cfg["embed"], depths=cfg["depths"],
                    num_heads=[3, 6, 12, 24], window_size=cfg["window"], mlp_ratio=4., drop_rate=0., attn_drop_rate=0.,
                    drop_path_rate=0.0, self_condition=True, symmetric_noise=False, out_chans_adj=cfg["c_e"],
                    out_chans_node=cfg["c_n"])
    net.load_state_dict(sd, strict=True)
    return net.to(DEV)


def _oracle_input_grads(cfg, sd, mode, adj, node, flags, noise, sc_adj, sc_node, wa, wn):
    a = adj.clone().requires_grad_(True)
    x = node.clone().requires_grad_(True)

    def net(aa, xx, f, c_noise, sa, sn):
        return O.denoiser_forward(sd, img=cfg["img"], embed=cfg["embed"], depths=cfg["depths"], heads=cfg["heads"],
                                  window=cfg["window"], self_condition=True, adj=aa, node=xx, flags=f, noise_labels=c_noise,
                                  sc_adj=sa, sc_node=sn)
    if mode == 0:
        da, dn = net(a, x, flags, noise, sc_adj, sc_node)
    else:
        da, dn = O.precond_forward(net, a, x, flags, noise, sc_adj, sc_node)
    ga, gx = torch.autograd.grad((da * wa).sum() + (dn * wn).sum(), (a, x))
    return ga, gx


_ORACLE = {}


def _case(name, mode):
    """Inputs, loss weights and the oracle's input gradients (cached: eval and training mode share them)."""
    key = (name, mode)
    if key not in _ORACLE:
        cfg = CONFIGS[name]
        batch = {"tiny": 4, "vg": 2, "coco": 4}[name]
        sd = synthetic_state_dict(cfg, seed=1234, stress=True)
        adj, node, flags, _, sc_adj, sc_node = synthetic_inputs(cfg, batch, seed=11)
        sigmas = torch.tensor([0.2, 1.5, 4.0, 0.7])[:batch].contiguous()
        noise = sigmas if mode == 1 else sigmas.log() / 4
        g = torch.Generator().manual_seed(5)
        wa, wn = torch.randn(adj.shape, generator=g), torch.randn(node.shape, generator=g)
        ref = _oracle_input_grads(cfg, sd, mode, adj, node, flags, noise, sc_adj, sc_node, wa, wn)
        _ORACLE[key] = (cfg, sd, (adj, node, flags, noise, sc_adj, sc_node), (wa, wn), ref)
    return _ORACLE[key]


def _native_input_grads(net, mode, inputs, weights, needs=(True, True)):
    adj, node, flags, noise, sc_adj, sc_node = (t.to(DEV) for t in inputs)
    a = adj.clone().requires_grad_(needs[0])
    x = node.clone().requires_grad_(needs[1])
    if mode == 0:
        da, dn = net(a, x, flags, noise, sc_adj, sc_node)
    else:
        model = NodeAdjPrecond(precond="edm", model=net, self_condition=False, symmetric_noise=False)   # no coin flip
        model.train(net.training)
        da, dn = model(a, x, flags, noise, sc_adj, sc_node)
    ((da * weights[0].to(DEV)).sum() + (dn * weights[1].to(DEV)).sum()).backward()
    torch.cuda.synchronize()
    return a.grad, x.grad


@pytest.mark.parametrize("training", [False, True])
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("name", ["tiny", "vg", "coco"])
def test_input_gradients_match_oracle_autograd(name, mode, training):
    cfg, sd, inputs, weights, (ref_a, ref_n) = _case(name, mode)
    net = _net(cfg, sd).train(training)
    ga, gn = _native_input_grads(net, mode, inputs, weights)
    assert ga is not None and gn is not None and torch.isfinite(ga).all() and torch.isfinite(gn).all()
    ea, en = _rel(ga, ref_a), _rel(gn, ref_n)
    print(f"INPUT_GRAD {name} mode {mode} {'train' if training else 'eval'}: d_adj {ea:.3e}, d_node {en:.3e}")
    # the parameter-gradient bound: bf16 GEMM operands in both directions (tests/test_gpu_train.py)
    assert ea < 4e-2 and en < 4e-2, (ea, en)
    params = dict(net.named_parameters())
    if training:
        assert all(p.grad is not None for p in params.values())
    else:
        assert all(p.grad is None for p in params.values())


# ---------------------------------------------------------------------------------------------------------
# side effects
# ---------------------------------------------------------------------------------------------------------
def _sampler(steps, graphs=True):
    s = NodeAdjEDMSampler(num_steps=steps, clip_samples=True, clip_samples_min=-1.0, clip_samples_max=1.0,
                          clip_samples_scope="x_0", dev=DEV, objective="edm", self_condition=True, symmetric_noise=False)
    s.use_graphs = graphs
    return s


def _seed(k):
    torch.manual_seed(k)
    torch.cuda.manual_seed(k)
    np.random.seed(k)


def test_eval_input_gradients_leave_parameters_and_sampling_alone():
    cfg, sd, inputs, weights, _ = _case("tiny", 1)
    net = _net(cfg, sd).eval()
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).eval()
    flags = inputs[2].to(DEV)
    kw = dict(num_node_chan=cfg["c_n"], num_edge_chan=cfg["c_e"])
    _seed(3)
    before = _sampler(6).sample(model, flags, **kw)
    w0 = {k: v.detach().clone() for k, v in net.state_dict().items()}
    ga, gn = _native_input_grads(net, 1, inputs, weights)
    assert ga is not None and gn is not None
    assert all(p.grad is None for p in net.parameters())
    assert all(torch.equal(w0[k], v) for k, v in net.state_dict().items())
    _seed(3)
    after = _sampler(6).sample(model, flags, **kw)
    assert torch.equal(before[0], after[0]) and torch.equal(before[1], after[1])


def test_training_parameter_gradients_do_not_depend_on_input_gradients():
    cfg, sd, inputs, weights, _ = _case("tiny", 1)
    grads = []
    for needs in ((False, False), (True, True)):
        net = _net(cfg, sd).train()
        _native_input_grads(net, 1, inputs, weights, needs)
        grads.append(torch.cat([p.grad.detach().flatten() for p in net.parameters()]))
    assert _rel(grads[1], grads[0]) < 1e-6, _rel(grads[1], grads[0])


@pytest.mark.parametrize("which", ["sigmas", "self_cond_x", "self_cond_feat"])
@pytest.mark.parametrize("training", [False, True])
def test_gradients_not_built_raise(which, training):
    cfg, sd, inputs, weights, _ = _case("tiny", 1)
    net = _net(cfg, sd).train(training)
    adj, node, flags, sig, sc_adj, sc_node = (t.to(DEV).clone() for t in inputs)
    adj.requires_grad_(True)
    {"sigmas": sig, "self_cond_x": sc_adj, "self_cond_feat": sc_node}[which].requires_grad_(True)
    da, dn = net.denoise(adj, node, flags, sig, sc_adj, sc_node)
    with pytest.raises(NotImplementedError, match=which.split("_")[0]):
        (da.sum() + dn.sum()).backward()


def test_double_backward_raises():
    cfg, sd, inputs, weights, _ = _case("tiny", 1)
    net = _net(cfg, sd).eval()
    adj, node, flags, sig, sc_adj, sc_node = (t.to(DEV) for t in inputs)
    a = adj.clone().requires_grad_(True)
    da, dn = net.denoise(a, node, flags, sig, sc_adj, sc_node)
    (g,) = torch.autograd.grad(da.sum() + dn.sum(), (a,), create_graph=True)
    with pytest.raises(RuntimeError):
        g.sum().backward()


# ---------------------------------------------------------------------------------------------------------
# guided completion
# ---------------------------------------------------------------------------------------------------------
def _tiny_model():
    cfg = CONFIGS["tiny"]
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    net = _net(cfg, sd).eval()
    return cfg, sd, NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).eval()


@pytest.mark.parametrize("graphs", [True, False])
def test_zero_guidance_is_sample_completion(graphs):
    cfg, _, model = _tiny_model()
    _, _, flags, _, _, _ = synthetic_inputs(cfg, 5, seed=9)
    flags = flags.to(DEV)
    n_adj, n_node = 5, 2
    g = torch.Generator().manual_seed(3)
    pick = flags.cpu() & (torch.rand(flags.shape, generator=g) < 0.5)
    node_cls = torch.where(pick, torch.randint(0, n_node, flags.shape, generator=g), -1)
    known = completion.encode_known(flags, cfg["c_e"], cfg["c_n"], node_cls, None, None, n_adj, n_node)
    kw = dict(num_node_chan=cfg["c_n"], num_edge_chan=cfg["c_e"])
    s = _sampler(6, graphs)
    _seed(4)
    a0, n0 = s.sample_completion(model, flags, *known, **kw)
    _seed(4)
    a1, n1 = s.sample_completion(model, flags, *known, guidance_scale=0.0, **kw)
    assert torch.equal(a0, a1) and torch.equal(n0, n1)


def test_guided_completion_matches_oracle_with_replayed_noise():
    """test_gpu_completion.py::test_completion_matches_oracle_with_replayed_noise with guidance: same noise, same coins,
    native vs guided_completion_oracle.sample(guidance=w); the oracle's guided and unguided results are further apart than the
    parity bound, and known entries of the final state are k exactly."""
    cfg, sd, model = _tiny_model()
    _, _, flags, _, _, _ = synthetic_inputs(cfg, 4, seed=7)
    steps, w = 8, 0.5
    ce, cn = cfg["c_e"], cfg["c_n"]
    g = torch.Generator().manual_seed(17)
    b, n = flags.shape
    pair = (flags[:, :, None] & flags[:, None, :])[:, None].expand(b, ce, n, n)
    ka = torch.where(pair & (torch.rand(b, ce, n, n, generator=g) < 0.5), torch.randn(b, ce, n, n, generator=g) * 2, NAN)
    kn = torch.where(flags[..., None] & (torch.rand(b, n, cn, generator=g) < 0.5), torch.randn(b, n, cn, generator=g) * 2,
                     NAN)
    ka, kn = torch.where(ka.isnan(), ka, ka.sign()), kn.clamp(-1, 1)
    log = []
    real_randn, real_like = torch.randn, torch.randn_like

    def rec_randn(*a, **k):
        t = real_randn(*a, **k)
        log.append(t.detach().cpu().clone())
        return t

    def rec_like(x, **k):
        t = real_like(x, **k)
        log.append(t.detach().cpu().clone())
        return t

    _seed(21)
    torch.randn, torch.randn_like = rec_randn, rec_like
    try:
        a, nd = _sampler(steps).sample_completion(model, flags.to(DEV), ka, kn, num_node_chan=cn, num_edge_chan=ce,
                                                  guidance_scale=w)
    finally:
        torch.randn, torch.randn_like = real_randn, real_like
    assert len(log) == 2 + 2 * steps

    def onet(adj, node, f, labels, sa, sn):
        return O.denoiser_forward(sd, img=cfg["img"], embed=cfg["embed"], depths=cfg["depths"], heads=cfg["heads"],
                                  window=cfg["window"], self_condition=cfg["self_cond"], adj=adj, node=node, flags=f,
                                  noise_labels=labels, sc_adj=sa, sc_node=sn)

    def omodel(aa, xx, f, sig, sa, sn):       # NodeAdjPrecond.forward: the coin-flip refresh is not differentiated
        if np.random.rand() < 0.5:
            with torch.no_grad():
                sa, sn = O.precond_forward(onet, aa, xx, f, sig, sa, sn)
        return O.precond_forward(onet, aa, xx, f, sig, sa, sn)

    def replay():
        it = iter(log)
        return lambda shape: next(it).reshape(shape)

    np.random.seed(21)
    with torch.no_grad():
        oa, on = GO.sample(omodel, flags, ce, cn, (ka, kn), num_steps=steps, normal=replay(), guidance=w)
    np.random.seed(21)
    with torch.no_grad():
        ua, un = CO.sample(omodel, flags, ce, cn, (ka, kn), num_steps=steps, normal=replay())
    fa, fn = ~ka.isnan(), ~kn.isnan()
    assert torch.equal(a[fa], ka[fa]) and torch.equal(nd[fn], kn[fn])
    assert torch.equal(oa[fa], ka[fa]) and torch.equal(on[fn], kn[fn])
    stats = dict(rel_adj=_rel(a, oa), rel_node=_rel(nd, on), guided_vs_unguided_adj=_rel(ua, oa),
                 guided_vs_unguided_node=_rel(un, on))
    print("GUIDED_COMPLETION_PARITY", stats)
    assert stats["rel_adj"] < 3e-2 and stats["rel_node"] < 3e-2, stats
    assert stats["guided_vs_unguided_adj"] > 3e-2 and stats["guided_vs_unguided_node"] > 3e-2, stats
