"""The oracle restatement must reproduce the unmodified reference (golden vectors)."""
import json
import os

import numpy as np
import pytest
import torch

from diffusesg_b200.utils.synthetic import CONFIGS, state_dict_spec, synthetic_inputs, synthetic_state_dict
from oracle import denoiser_oracle as O
from oracle import edm_oracle as E


def _net(cfg, sd):
    def f(adj, node, flags, labels, sa, sn):
        return O.denoiser_forward(sd, img=cfg["img"], embed=cfg["embed"], depths=cfg["depths"], heads=cfg["heads"],
                                  window=cfg["window"], self_condition=cfg["self_cond"], adj=adj, node=node,
                                  flags=flags, noise_labels=labels, sc_adj=sa, sc_node=sn)
    return f


@pytest.mark.parametrize("name", ["vg", "coco", "tiny", "n64w16"])
def test_state_dict_layout_matches_reference(name, golden_dir):
    ref = json.load(open(os.path.join(golden_dir, f"layout_{name}.json")))
    spec = state_dict_spec(CONFIGS[name])
    assert [k for k, _, _ in ref["layout"]] == list(spec.keys())
    for (k, shape, _), (shape2, _) in zip(ref["layout"], spec.values()):
        assert tuple(shape) == tuple(shape2), k


@pytest.mark.parametrize("name,batch", [("tiny", 3), ("vg", 2), ("coco", 2)])
def test_forward_matches_reference(name, batch, golden_dir):
    torch.set_num_threads(8)
    cfg = CONFIGS[name]
    g = np.load(os.path.join(golden_dir, f"forward_{name}.npz"))
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    adj, node, flags, sigmas, sc_adj, sc_node = synthetic_inputs(cfg, batch, seed=7)
    labels = torch.from_numpy(g["labels"])
    net = _net(cfg, sd)
    with torch.no_grad():
        a, n = net(adj, node, flags, labels, sc_adj, sc_node)
        a0, n0 = net(adj, node, flags, labels, None, None)
    # identical op sequence in fp32; the only slack is GEMM blocking order
    for got, key in ((a, "adj_sc"), (n, "node_sc"), (a0, "adj_nosc"), (n0, "node_nosc")):
        want = torch.from_numpy(g[key])
        rel = (got - want).norm() / want.norm()
        assert rel < 2e-6, (key, float(rel))
    assert float(torch.from_numpy(g["adj_sc"]).abs().mean()) > 1e-2   # stress init makes the output visible


def test_precond_matches_reference(golden_dir):
    cfg = CONFIGS["tiny"]
    g = np.load(os.path.join(golden_dir, "precond_tiny.npz"))
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    adj, node, flags, _, _, _ = synthetic_inputs(cfg, 3, seed=7)
    coins = iter(g["coins"])
    sa = sn = None
    with torch.no_grad():
        for k, s in enumerate((40.0, 3.0, 0.4, 0.01)):
            sa, sn = O.precond_forward(_net(cfg, sd), adj * s, node * s, flags, torch.full((3,), s), sa, sn,
                                       coin=lambda: next(coins))
            for got, key in ((sa, f"adj_{k}"), (sn, f"node_{k}")):
                want = torch.from_numpy(g[key])
                assert (got - want).norm() / want.norm() < 2e-6, key


def test_sampler_matches_reference(golden_dir):
    cfg = CONFIGS["tiny"]
    g = np.load(os.path.join(golden_dir, "sampler_tiny.npz"))
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    _, _, flags, _, _, _ = synthetic_inputs(cfg, 3, seed=7)
    flags = flags[:2]
    np.testing.assert_array_equal(E.t_steps_fp32(8).numpy(), g["t_steps"])
    np.testing.assert_array_equal(E.sigma_grid(256).numpy(), g["sigma_steps_256"])

    def model(a, n, f, sig, sa, sn):
        return O.precond_forward(_net(cfg, sd), a, n, f, sig, sa, sn, coin=np.random.rand)

    torch.manual_seed(11)
    np.random.seed(11)
    trace = []
    with torch.no_grad():
        a, n = E.sample(model, flags, cfg["c_e"], cfg["c_n"], num_steps=8, trace=trace)
    assert (a - torch.from_numpy(g["adjs"])).abs().max() < 2e-4
    assert (n - torch.from_numpy(g["nodes"])).abs().max() < 2e-4
    # interim snapshots of the reference: init + steps linspace(0, 8, 4).astype(int).clip(max=7) = 0, 2, 5, 7
    for slot, step in zip(range(1, 5), (0, 2, 5, 7)):
        assert (trace[step][1] - torch.from_numpy(g["nodes_ls"][slot])).abs().max() < 2e-4


def test_sampler_known_answer(golden_dir):
    """The reference's own KAT (sanity_check_gt_*): the last Euler step returns the ground truth."""
    g = np.load(os.path.join(golden_dir, "sampler_tiny.npz"))
    cfg = CONFIGS["tiny"]
    _, _, flags, _, _, _ = synthetic_inputs(cfg, 3, seed=7)
    gt = (torch.from_numpy(g["kat_gt_adjs"]), torch.from_numpy(g["kat_gt_nodes"]))
    torch.manual_seed(12)
    a, n = E.sample(None, flags[:2], cfg["c_e"], cfg["c_n"], num_steps=8, gt=gt)
    np.testing.assert_array_equal(a.numpy(), g["kat_adjs"])
    np.testing.assert_array_equal(n.numpy(), g["kat_nodes"])
    assert (a - gt[0]).abs().max() < 1e-6 and (n - gt[1]).abs().max() < 1e-6


def test_training_objective_and_loss_match_reference(golden_dir):
    """oracle/train_oracle.py against the unmodified reference's NodeAdjEDMObjectiveGenerator / NodeAdjRainbowLoss
    (SURVEY 8a row a17): bit-exact noising and coefficients, loss within fp32 summation-order slack."""
    from oracle import train_oracle as T
    g = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(golden_dir, "train_objective.npz")).items()}
    _, _, flags, _, _, _ = synthetic_inputs(CONFIGS["tiny"], 4, seed=7)
    sigmas, weights = T.training_sigmas_weights(g["rnd"])
    assert torch.equal(sigmas, g["sigmas"]) and torch.equal(weights, g["weights"])
    in_a, _, in_x, _ = T.network_input(g["clean_a"], g["clean_x"], flags, sigmas, g["eps_a"], g["eps_x"])
    assert torch.equal(in_a, g["in_a"]) and torch.equal(in_x, g["in_x"])
    for red in ("none", "mean"):
        la, ln = T.regression_loss(g["pred_a"], g["pred_x"], g["clean_a"], g["clean_x"], flags, weights, 1.0, 0.5, red)
        torch.testing.assert_close(la, g[f"loss_adj_{red}"], rtol=1e-6, atol=0)
        torch.testing.assert_close(ln, g[f"loss_node_{red}"], rtol=1e-6, atol=0)


@pytest.mark.parametrize("name", ["vg", "coco"])
def test_precond_matches_reference_full_geometries(name, golden_dir):
    """NodeAdjPrecond.forward of the unmodified reference on the shipped geometries (coin-flip stream included)."""
    torch.set_num_threads(8)
    cfg = CONFIGS[name]
    g = np.load(os.path.join(golden_dir, f"precond_{name}.npz"))
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    adj, node, flags, _, _, _ = synthetic_inputs(cfg, 2, seed=7)
    coins = iter(g["coins"])
    sa = sn = None
    with torch.no_grad():
        for k, s in enumerate((40.0, 3.0, 0.4, 0.01)):
            sa, sn = O.precond_forward(_net(cfg, sd), adj * s, node * s, flags, torch.full((2,), s), sa, sn,
                                       coin=lambda: next(coins))
            for got, key in ((sa, f"adj_{k}"), (sn, f"node_{k}")):
                want = torch.from_numpy(g[key])
                assert (got - want).norm() / want.norm() < 2e-6, key


RAW_TYPES = {"vg": (150, 51), "coco": (171, 7)}   # raw_num_node_type, raw_num_adj_type (utils/sg_utils.py:355-394)


@pytest.mark.parametrize("name", ["vg", "coco"])
def test_decode_matches_reference_closures(name, golden_dir):
    """oracle.edm_oracle.decode_samples against the reference's own _decode_node / _decode_adj (the closures of
    sg_go_sampling, runner/sampler/sampler_node_adj.py:222-285, executed from their source text by
    tests/golden/make_golden_full.py) and its bbox rule (:202-209): bit-exact, on the 256-step samples of the
    reference and on an edge-case tensor (exact zeros, values beyond the clamp, out-of-range bit patterns)."""
    g = np.load(os.path.join(golden_dir, f"decode_{name}.npz"))
    s = np.load(os.path.join(golden_dir, f"sampler256_{name}.npz"))
    n_node, n_adj = RAW_TYPES[name]
    cases = {"final": (s["adjs"], s["nodes"], s["flags"]), "edge": (g["edge_adj"], g["edge_node"], g["edge_flags"])}
    for key, (a, n, f) in cases.items():
        qa, qn, box = E.decode_samples(torch.from_numpy(a), torch.from_numpy(n), torch.from_numpy(f), n_adj, n_node)
        np.testing.assert_array_equal(qa.numpy(), g[f"{key}_q_adj"])
        np.testing.assert_array_equal(qn.numpy(), g[f"{key}_q_node"])
        np.testing.assert_array_equal(box.numpy(), g[f"{key}_bbox"])
    assert g["edge_q_adj"].max() == n_adj - 1 and g["edge_q_node"].max() == n_node - 1   # the clamp is exercised


def _cpu_stream_normal(shape):
    return torch.randn(shape)


@pytest.mark.parametrize("case,name", [("coco", "coco"), ("vg", "vg")])
def test_sampler256_first_snapshot_matches_reference(case, name, sampler256_golden):
    """The oracle loop on the 256-step schedule against the reference's 256-step golden run, through the first
    interim snapshot (after step 0; the full-length comparison is DSG_SLOW=1 / tools, it takes minutes on a CPU).
    Noise and coins come from the global generators seeded like the golden run."""
    torch.set_num_threads(8)
    cfg = CONFIGS[name]
    g = sampler256_golden(case)
    steps = 256 if os.environ.get("DSG_SLOW", "0") == "1" else 1
    sd = synthetic_state_dict(cfg, seed=1234, stress=(case != "vg_refinit"))
    flags = torch.from_numpy(g["flags"])

    def model(a, n, f, sig, sa, sn):
        return O.precond_forward(_net(cfg, sd), a, n, f, sig, sa, sn, coin=np.random.rand)

    torch.manual_seed(int(g["torch_seed"]))
    np.random.seed(int(g["numpy_seed"]))
    ts = E.t_steps_fp32(256)
    with torch.no_grad():
        adjs, nodes = E.init_sample(flags, cfg["c_e"], cfg["c_n"], _cpu_stream_normal)
        np.testing.assert_array_equal(nodes[:2].numpy(), g["nodes_ls"][0])          # the initial noise itself
        adjs, nodes = adjs * ts[0], nodes * ts[0]
        sc_a = sc_n = None
        snap = {int(s): k + 1 for k, s in enumerate(g["snapshot_steps"])}
        for i in range(steps):
            adjs, nodes, sc_a, sc_n, _ = E.heun_step(model, adjs, nodes, flags, sc_a, sc_n, ts[i], ts[i + 1], i, 256,
                                                     _cpu_stream_normal)
            if i in snap:
                for got, want in ((adjs[:2], g["adjs_ls"][snap[i]]), (nodes[:2], g["nodes_ls"][snap[i]])):
                    want = torch.from_numpy(want)
                    assert (got - want).norm() / want.norm() < 1e-5, (i, float((got - want).norm() / want.norm()))
    if steps == 256:
        assert (adjs - torch.from_numpy(g["adjs"])).norm() / torch.from_numpy(g["adjs"]).norm() < 1e-4


def _train_case(cfg, batch):
    """The inputs tests/golden/make_golden_train.py fed the unmodified reference (same construction, restated here)."""
    adj, node, flags, _, sc_adj, sc_node = synthetic_inputs(cfg, batch, seed=11)
    sigmas = torch.tensor([0.2, 1.5, 4.0, 0.7, 0.05, 9.0, 0.9, 2.2])[:batch].contiguous()
    f = flags.float()
    tgt_adj = adj.sign() * f[:, None, :, None] * f[:, None, None, :]
    tgt_node = node.clamp(-1, 1) * f[:, :, None]
    weights = (sigmas ** 2 + 0.25) / (sigmas * 0.5) ** 2
    return adj, node, flags, sigmas, sc_adj, sc_node, tgt_adj, tgt_node, weights


@pytest.mark.parametrize("name,batch", [("tiny", 4), ("vg", 2)])
def test_training_gradients_match_reference(name, batch, golden_dir):
    """One training iteration's forward + backward (trainer_node_adj.py:104-173) on the oracle with torch autograd against
    the gradients the UNMODIFIED reference produced (tests/golden/train_grads_*.npz): pins what the GPU gradient-parity
    tests of the native backward compare with."""
    from oracle import train_oracle as T
    torch.set_num_threads(8)
    cfg = CONFIGS[name]
    g = np.load(os.path.join(golden_dir, f"train_grads_{name}.npz"))
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    leaves = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "attn_mask" not in k else v) for k, v in sd.items()}
    adj, node, flags, sigmas, sc_adj, sc_node, tgt_adj, tgt_node, weights = _train_case(cfg, batch)
    da, dn = O.precond_forward(_net(cfg, leaves), adj, node, flags, sigmas, sc_adj, sc_node)
    la, ln = T.regression_loss(da, dn, tgt_adj, tgt_node, flags, weights, 1.0, 1.0, "none")
    (la.mean() + ln.mean()).backward()
    assert np.allclose(la.detach().numpy(), g["loss_adj"], rtol=1e-5) and np.allclose(ln.detach().numpy(), g["loss_node"], rtol=1e-5)
    keys, norms = list(g["keys"]), g["norms"]
    assert len(keys) == sum(1 for v in leaves.values() if v.is_floating_point() and v.requires_grad)
    for k, want in zip(keys, norms):
        got = float(leaves[k].grad.double().norm())
        assert abs(got - want) <= 2e-4 * max(want, 1e-6 * norms.max()), (k, got, want)
    for key in g.files:
        if key.startswith("grad::"):
            want = torch.from_numpy(g[key])
            got = leaves[key[6:]].grad
            assert float((got - want).norm() / want.norm().clamp_min(1e-20)) < 1e-4, key
