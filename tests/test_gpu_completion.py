"""Scene-graph completion on the B200: the completion kernels bit-exact against their fp32 torch expressions, and
NodeAdjEDMSampler.sample_completion against sample(), the oracle, itself under CUDA graphs and under padding
skipping (DESIGN.md §3.6)."""
import numpy as np
import pytest
import torch

from diffusesg_b200 import native
from diffusesg_b200.model.diffusesg.diffusesg import DiffuseSG
from diffusesg_b200.model.precond.precond import NodeAdjPrecond
from diffusesg_b200.runner.mcmc_sampler import completion
from diffusesg_b200.runner.mcmc_sampler.edm import NodeAdjEDMSampler
from diffusesg_b200.utils.synthetic import CONFIGS, in_chans, synthetic_inputs, synthetic_state_dict
from oracle import denoiser_oracle as O
from oracle import completion_oracle as CO
from oracle import edm_oracle as E
from oracle.denoiser_oracle import mask_pairs, mask_rows

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
NAN = float("nan")
# (num_adj_type, num_node_type) per geometry: the VG dataset counts, and counts that fit the bits of tiny / COCO
TYPES = {"tiny": (5, 2), "vg": (51, 150), "coco": (7, 171)}


def build(cfg, stress=True):
    m = DiffuseSG(img_size=cfg["img"], in_chans=in_chans(cfg), patch_size=1, embed_dim=cfg["embed"],
                  depths=cfg["depths"], num_heads=[3, 6, 12, 24], window_size=cfg["window"], mlp_ratio=4.,
                  drop_rate=0., attn_drop_rate=0., drop_path_rate=0.0, self_condition=cfg["self_cond"],
                  symmetric_noise=False, out_chans_adj=cfg["c_e"], out_chans_node=cfg["c_n"])
    sd = synthetic_state_dict(cfg, seed=1234, stress=stress)
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval(), sd


def precond(net):
    return NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).eval()


def make_sampler(steps, graphs=True, eager_every=0, skip=True):
    s = NodeAdjEDMSampler(num_steps=steps, clip_samples=True, clip_samples_min=-1.0, clip_samples_max=1.0,
                          clip_samples_scope="x_0", dev=DEV, objective="edm", self_condition=True, symmetric_noise=False)
    s.use_graphs, s.eager_every, s.skip_padding = graphs, eager_every, skip
    return s


def seed(k):
    torch.manual_seed(k)
    torch.cuda.manual_seed(k)
    np.random.seed(k)


def flags_with_counts(cfg, counts):
    return torch.arange(cfg["img"])[None, :] < torch.tensor(counts)[:, None]


def conditions(flags, n_adj, n_node, seed_, frac=0.5):
    """About `frac` of the valid nodes with class and box known, plus every relation among the known nodes."""
    g = torch.Generator().manual_seed(seed_)
    b, n = flags.shape
    pick = flags & (torch.rand(b, n, generator=g) < frac)
    node_cls = torch.where(pick, torch.randint(0, n_node, (b, n), generator=g), torch.full((b, n), -1))
    bbox = torch.where(pick[..., None], torch.rand(b, n, 4, generator=g), torch.full((b, n, 4), NAN))
    pair = pick[:, :, None] & pick[:, None, :] & ~torch.eye(n, dtype=torch.bool)
    adj_cls = torch.where(pair, torch.randint(0, n_adj, (b, n, n), generator=g), torch.full((b, n, n), -1))
    return node_cls, bbox, adj_cls


def free_condition(b, ce, n, cn):
    return torch.full((b, ce, n, n), NAN, device=DEV), torch.full((b, n, cn), NAN, device=DEV)


def random_known(flags, ce, cn, g, frac=0.5):
    """Raw NaN-coded state: about `frac` of the valid entries known (arbitrary finite values)."""
    b, n = flags.shape
    pair = (flags[:, :, None] & flags[:, None, :])[:, None].expand(b, ce, n, n)
    ka = torch.where(pair & (torch.rand(b, ce, n, n, generator=g) < frac), torch.randn(b, ce, n, n, generator=g) * 2, NAN)
    kn = torch.where(flags[..., None] & (torch.rand(b, n, cn, generator=g) < frac), torch.randn(b, n, cn, generator=g) * 2,
                     NAN)
    return ka, kn


def where_pre(x, eps, k, c, t_hat, flags, adj):
    out = torch.where(k.isnan(), x + c * eps, k + t_hat * eps)
    return mask_pairs(out, flags) if adj else mask_rows(out, flags)


# ---------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("b,ce,n,cn", [(3, 3, 16, 5), (8, 6, 64, 12), (512, 6, 64, 12), (5, 3, 40, 12), (1, 1, 4, 1),
                                       (700, 3, 40, 12)])
def test_pre_step_known_kernels_match_torch(b, ce, n, cn):
    """Both completion pre-steps == torch.where(k.isnan(), x + c eps, k + t_hat eps), masked, bit for bit; the Philox
    one with eps = randn_like(adj), randn_like(node) at the same generator state, which it advances the same way."""
    g = torch.Generator().manual_seed(b * 7 + n)
    flags = torch.arange(n)[None, :] < torch.randint(1, n + 1, (b, 1), generator=g)
    adj, node = torch.randn(b, ce, n, n, generator=g) * 3, torch.randn(b, n, cn, generator=g) * 3
    ka, kn = random_known(flags, ce, cn, g)
    s = E.step_scalars(E.t_steps_fp32(256)[40], E.t_steps_fp32(256)[41], 256)
    c, t_hat = s["noise_coef"], s["t_hat"]
    cu = lambda t: t.to(DEV)
    known = (cu(ka), cu(kn))
    # caller-drawn noise
    eps_a, eps_n = torch.randn(b, ce, n, n, generator=g), torch.randn(b, n, cn, generator=g)
    ga, gn = native.edm_pre_step_known(cu(adj), cu(node), cu(eps_a), cu(eps_n), known, cu(flags), float(c), float(t_hat))
    np.testing.assert_array_equal(ga.cpu().numpy(), where_pre(adj, eps_a, ka, c, t_hat, flags, True).numpy())
    np.testing.assert_array_equal(gn.cpu().numpy(), where_pre(node, eps_n, kn, c, t_hat, flags, False).numpy())
    # in-kernel Philox noise
    for sd, burn in ((1234, 0), (99, 3)):
        torch.cuda.manual_seed(sd)
        for _ in range(burn):
            torch.randn(1000, device=DEV)
        ea, en = torch.randn_like(cu(adj)), torch.randn_like(cu(node))
        next_want = torch.randn(4097, device=DEV)
        torch.cuda.manual_seed(sd)
        for _ in range(burn):
            torch.randn(1000, device=DEV)
        fa, fn = native.edm_pre_step_fused_noise_known(cu(adj), cu(node), known, cu(flags), float(c), float(t_hat))
        next_got = torch.randn(4097, device=DEV)
        np.testing.assert_array_equal(fa.cpu().numpy(), where_pre(adj, ea.cpu(), ka, c, t_hat, flags, True).numpy())
        np.testing.assert_array_equal(fn.cpu().numpy(), where_pre(node, en.cpu(), kn, c, t_hat, flags, False).numpy())
        assert torch.equal(next_got, next_want)
    # an all-free condition is the plain pre-step
    fr = (torch.full_like(known[0], NAN), torch.full_like(known[1], NAN))
    pa, pn = native.edm_pre_step(cu(adj), cu(node), cu(eps_a), cu(eps_n), cu(flags), float(c))
    qa, qn = native.edm_pre_step_known(cu(adj), cu(node), cu(eps_a), cu(eps_n), fr, cu(flags), float(c), float(t_hat))
    assert torch.equal(pa, qa) and torch.equal(pn, qn)


@pytest.mark.parametrize("b,ce,n,cn", [(3, 3, 16, 5), (8, 6, 64, 12), (5, 3, 40, 12), (1, 1, 4, 1)])
def test_apply_known_bit_exact(b, ce, n, cn):
    g = torch.Generator().manual_seed(3 * b + n)
    flags = torch.arange(n)[None, :] < torch.randint(1, n + 1, (b, 1), generator=g)
    adj, node = mask_pairs(torch.randn(b, ce, n, n, generator=g), flags), mask_rows(torch.randn(b, n, cn, generator=g), flags)
    ka, kn = random_known(flags, ce, cn, g)
    xa, xn = adj.to(DEV), node.to(DEV)
    native.edm_apply_known(xa, xn, (ka.to(DEV), kn.to(DEV)), flags.to(DEV))
    np.testing.assert_array_equal(xa.cpu().numpy(), mask_pairs(torch.where(ka.isnan(), adj, ka), flags).numpy())
    np.testing.assert_array_equal(xn.cpu().numpy(), mask_rows(torch.where(kn.isnan(), node, kn), flags).numpy())


@pytest.mark.parametrize("name", ["tiny", "vg", "coco"])
def test_encode_known_inverts_decode(name):
    """encode_known (device) == the oracle's encoder bit for bit; dsg_decode_samples of it gives back the classes, and
    the boxes as the fp32 (2 b - 1) * 0.5 + 0.5."""
    cfg = CONFIGS[name]
    ce, cn = cfg["c_e"], cfg["c_n"]
    n_adj, n_node = TYPES[name]
    flags = flags_with_counts(cfg, [cfg["allowed_nodes"], 3, 1, cfg["img"] // 2])
    node_cls, bbox, adj_cls = conditions(flags, n_adj, n_node, 21, frac=0.7)
    adj_cls[0, 0, 1] = 0                                                 # class 0 ("no relation") is a constraint
    ka, kn = completion.encode_known(flags.to(DEV), ce, cn, node_cls, bbox, adj_cls, n_adj, n_node)
    oa, on = CO.encode_known(flags, ce, cn, node_cls, bbox, adj_cls)
    np.testing.assert_array_equal(ka.cpu().numpy(), oa.numpy())
    np.testing.assert_array_equal(kn.cpu().numpy(), on.numpy())
    qa, qn, qb = native.decode_samples(ka, kn, flags.to(DEV), n_adj, n_node)
    on_n, on_a = node_cls >= 0, adj_cls >= 0
    assert torch.equal(qn.cpu().long()[on_n], node_cls[on_n]) and torch.equal(qa.cpu().long()[on_a], adj_cls[on_a])
    want_box = (2.0 * bbox - 1.0) * 0.5 + 0.5
    np.testing.assert_array_equal(qb.cpu()[on_n].numpy(), want_box[on_n].numpy())
    # nothing given: everything free
    fa, fn = completion.encode_known(flags.to(DEV), ce, cn)
    assert bool(fa.isnan().all()) and bool(fn.isnan().all())


# ---------------------------------------------------------------------------------------------------------
# sampler
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("graphs,eager_every", [(False, 0), (True, 0), (True, 3)])
def test_empty_condition_is_a_no_op(graphs, eager_every):
    """sample_completion with an all-NaN condition == sample() and == sample_decoded(): same samples, same generator
    state afterwards, same denoiser pass count."""
    cfg = CONFIGS["tiny"]
    net, _ = build(cfg)
    model = precond(net)
    _, _, flags, _, _, _ = synthetic_inputs(cfg, 6, seed=9)
    flags = flags.to(DEV)
    ce, cn = cfg["c_e"], cfg["c_n"]
    n_adj, n_node = TYPES["tiny"]
    free = free_condition(6, ce, cfg["img"], cn)
    sampler = make_sampler(7, graphs, eager_every)
    outs = {}
    for kind in ("sample", "completion", "decoded", "completion_decoded", "completion_again"):
        seed(5)
        if kind == "sample":
            r = sampler.sample(model=model, node_flags=flags, num_node_chan=cn, num_edge_chan=ce)
        elif kind == "decoded":
            r = sampler.sample_decoded(model, flags, n_adj, n_node, num_node_chan=cn, num_edge_chan=ce)
        elif kind == "completion_decoded":
            r = sampler.sample_completion(model, flags, *free, num_node_chan=cn, num_edge_chan=ce, decode=(n_adj, n_node))
        else:
            r = sampler.sample_completion(model, flags, *free, num_node_chan=cn, num_edge_chan=ce)
        outs[kind] = (tuple(r), torch.randn(100, device=DEV).cpu(), sampler.last_raw_passes)
    for a, b in (("sample", "completion"), ("decoded", "completion_decoded"), ("sample", "completion_again")):
        (ra, ga, pa), (rb, gb, pb) = outs[a], outs[b]
        assert all(torch.equal(x, y) for x, y in zip(ra, rb)), (a, b)
        assert torch.equal(ga, gb) and pa == pb, (a, b)
    assert outs["sample"][2] >= 2 * 7 - 1


@pytest.mark.parametrize("name,counts", [("tiny", [14, 9, 5, 12]), ("vg", [62, 17, 33, 5]), ("coco", [33, 11, 21, 2])])
def test_known_entries_are_held(name, counts):
    cfg = CONFIGS[name]
    net, _ = build(cfg, stress=False)
    model = precond(net)
    ce, cn = cfg["c_e"], cfg["c_n"]
    n_adj, n_node = TYPES[name]
    flags = flags_with_counts(cfg, counts)
    node_cls, bbox, adj_cls = conditions(flags, n_adj, n_node, 31)
    known = completion.encode_known(flags.to(DEV), ce, cn, node_cls, bbox, adj_cls, n_adj, n_node)
    sampler = make_sampler(4)
    kw = dict(num_node_chan=cn, num_edge_chan=ce)
    seed(7)
    a, n = sampler.sample_completion(model, flags.to(DEV), *known, **kw)
    seed(7)
    qa, qn, qb = sampler.sample_completion(model, flags.to(DEV), *known, decode=(n_adj, n_node), **kw)
    seed(7)
    a0, n0 = sampler.sample_completion(model, flags.to(DEV), *free_condition(len(counts), ce, cfg["img"], cn), **kw)
    ka, kn = known[0].cpu(), known[1].cpu()
    fa, fn = ~ka.isnan(), ~kn.isnan()
    assert int(fa.sum()) > 0 and int(fn.sum()) > 0
    assert torch.equal(a[fa], ka[fa]) and torch.equal(n[fn], kn[fn])
    on_n, on_a = node_cls >= 0, adj_cls >= 0
    assert torch.equal(qn.long()[on_n], node_cls[on_n]) and torch.equal(qa.long()[on_a], adj_cls[on_a])
    np.testing.assert_array_equal(qb[on_n].numpy(), ((2.0 * bbox - 1.0) * 0.5 + 0.5)[on_n].numpy())
    pair = (flags[:, None, :, None] & flags[:, None, None, :]).expand_as(a)
    assert not torch.equal(a[~fa & pair], a0[~fa & pair])
    assert not torch.equal(n[~fn & flags[..., None].expand_as(n)], n0[~fn & flags[..., None].expand_as(n)])
    assert float(a[~pair].abs().sum()) == 0.0 and float(n[~flags].abs().sum()) == 0.0


def _replay(noise_log):
    it = iter(noise_log)
    return lambda shape: next(it).reshape(shape)


def test_completion_matches_oracle_with_replayed_noise():
    """test_gpu_denoiser.py::test_sampler_matches_oracle_with_replayed_noise with about half the entries known: same
    noise, same coins, native vs completion_oracle.sample driving the oracle network; known entries agree exactly."""
    cfg = CONFIGS["tiny"]
    net, sd = build(cfg)
    model = precond(net)
    _, _, flags, _, _, _ = synthetic_inputs(cfg, 4, seed=7)
    steps = 8
    ce, cn = cfg["c_e"], cfg["c_n"]
    ka, kn = random_known(flags, ce, cn, torch.Generator().manual_seed(17))
    ka, kn = torch.where(ka.isnan(), ka, ka.sign()), kn.clamp(-1, 1)   # clean-data range (torch.sign(NaN) is 0)
    sampler = make_sampler(steps)
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

    seed(21)
    torch.randn, torch.randn_like = rec_randn, rec_like
    try:
        a, n = sampler.sample_completion(model, flags.to(DEV), ka, kn, num_node_chan=cn, num_edge_chan=ce)
    finally:
        torch.randn, torch.randn_like = real_randn, real_like
    assert len(log) == 2 + 2 * steps
    np.random.seed(21)

    def onet(adj, node, f, labels, sa, sn):
        return O.denoiser_forward(sd, img=cfg["img"], embed=cfg["embed"], depths=cfg["depths"], heads=cfg["heads"],
                                  window=cfg["window"], self_condition=cfg["self_cond"], adj=adj, node=node, flags=f,
                                  noise_labels=labels, sc_adj=sa, sc_node=sn)

    omodel = lambda aa, nn_, f, sig, sa, sn: O.precond_forward(onet, aa, nn_, f, sig, sa, sn, coin=np.random.rand)
    with torch.no_grad():
        oa, on = CO.sample(omodel, flags, ce, cn, (ka, kn), num_steps=steps, normal=_replay(log))
    fa, fn = ~ka.isnan(), ~kn.isnan()
    assert torch.equal(a[fa], ka[fa]) and torch.equal(oa[fa], ka[fa])
    assert torch.equal(n[fn], kn[fn]) and torch.equal(on[fn], kn[fn])
    rel = lambda x, y: float((x.double() - y.double()).norm() / y.double().norm())
    valid_pair = flags[:, :, None] & flags[:, None, :]
    nb = cn - 4
    edge_g, edge_o = E.decode_bits(a.permute(0, 2, 3, 1), 2 ** ce), E.decode_bits(oa.permute(0, 2, 3, 1), 2 ** ce)
    node_g, node_o = E.decode_bits(n[..., :nb], 2 ** nb), E.decode_bits(on[..., :nb], 2 ** nb)
    stats = dict(rel_adj=rel(a, oa), rel_node=rel(n, on), edge_agree=float((edge_g == edge_o)[valid_pair].float().mean()),
                 node_agree=float((node_g == node_o)[flags].float().mean()), known=(int(fa.sum()), int(fn.sum())))
    print("COMPLETION_PARITY", stats)
    assert stats["rel_adj"] < 3e-2 and stats["rel_node"] < 3e-2, stats
    assert stats["edge_agree"] >= 0.95 and stats["node_agree"] >= 0.95, stats
    far_e = (oa.abs() > 0.06).permute(0, 2, 3, 1).all(-1) & valid_pair
    far_n = (on[..., :nb].abs() > 0.06).all(-1) & flags
    assert bool((edge_g == edge_o)[far_e].all()) and bool((node_g == node_o)[far_n].all()), stats


def test_completion_graphs_match_eager():
    """Completion under CUDA graphs (also with every 3rd step eager) == the eager loop, bit for bit, decoded too."""
    cfg = CONFIGS["tiny"]
    net, _ = build(cfg)
    model = precond(net)
    _, _, flags, _, _, _ = synthetic_inputs(cfg, 6, seed=9)
    flags = flags.to(DEV)
    ce, cn = cfg["c_e"], cfg["c_n"]
    known = completion.encode_known(flags, ce, cn, *conditions(flags.cpu(), *TYPES["tiny"], 41), *TYPES["tiny"])
    outs = []
    for graphs, eager_every in ((False, 0), (True, 0), (True, 3)):
        sampler = make_sampler(10, graphs, eager_every)
        res = []
        for decode in (None, TYPES["tiny"], None):
            seed(5)
            res += list(sampler.sample_completion(model, flags, *known, num_node_chan=cn, num_edge_chan=ce, decode=decode))
            res.append(torch.randn(100, device=DEV).cpu())
            res.append(torch.tensor(sampler.last_raw_passes))
        assert (sampler._plan is not None) == graphs
        outs.append(res)
    for o in outs[1:]:
        assert len(o) == len(outs[0]) and all(torch.equal(x, y) for x, y in zip(outs[0], o))


def test_graphs_interleave_sample_and_completion():
    """One sampler (graphs, padding skipping): sample -> sample_completion -> sample -> sample_completion with a
    different condition each time == fresh eager samplers for each call: the graph key keeps the two kinds apart and
    the condition buffer is refilled per run."""
    cfg = CONFIGS["vg"]
    net, _ = build(cfg, stress=False)
    model = precond(net)
    ce, cn = cfg["c_e"], cfg["c_n"]
    flags = flags_with_counts(cfg, [5, 17, 33, 62, 20, 48]).to(DEV)
    conds = [None, completion.encode_known(flags, ce, cn, *conditions(flags.cpu(), 51, 150, 50), 51, 150), None,
             completion.encode_known(flags, ce, cn, *conditions(flags.cpu(), 51, 150, 51, frac=0.3), 51, 150)]
    shared = make_sampler(3)

    def run(sampler, k, cond):
        seed(60 + k)
        if cond is None:
            return sampler.sample(model=model, node_flags=flags, num_node_chan=cn, num_edge_chan=ce)
        return sampler.sample_completion(model, flags, *cond, num_node_chan=cn, num_edge_chan=ce)

    got = [run(shared, k, c) for k, c in enumerate(conds)]
    want = [run(make_sampler(3, graphs=False), k, c) for k, c in enumerate(conds)]
    for (a0, n0), (a1, n1) in zip(got, want):
        assert torch.equal(a0, a1) and torch.equal(n0, n1)
    assert not torch.equal(got[1][0], got[3][0])


@pytest.mark.parametrize("counts", [[2, 9, 16, 17, 33, 48, 62, 5], [30] * 5])
def test_completion_padding_skipping_matches_dense(counts):
    """Known entries lie on valid pairs only, so the padded inputs the compact schedule skips stay zero: completion
    with padding skipping == the dense schedule, bit for bit."""
    cfg = CONFIGS["vg"]
    net, _ = build(cfg, stress=False)
    model = precond(net)
    ce, cn = cfg["c_e"], cfg["c_n"]
    flags = flags_with_counts(cfg, counts)
    flags[0, 0] = False
    known = completion.encode_known(flags.to(DEV), ce, cn, *conditions(flags, 51, 150, 70), 51, 150)
    outs = []
    for skip in (True, False):
        sampler = make_sampler(3, skip=skip)
        seed(8)
        outs.append(sampler.sample_completion(model, flags.to(DEV), *known, num_node_chan=cn, num_edge_chan=ce))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
