"""Scene-graph completion without a GPU: the oracle's completion rules, its encoder, and the input checks of
runner/mcmc_sampler/completion.py and NodeAdjEDMSampler.sample_completion (all of which run before any kernel)."""
import numpy as np
import pytest
import torch

from diffusesg_b200 import native
from diffusesg_b200.runner.mcmc_sampler import completion
from diffusesg_b200.runner.mcmc_sampler.edm import NodeAdjEDMSampler
from diffusesg_b200.utils.synthetic import CONFIGS, synthetic_node_flags
from oracle import completion_oracle as CO
from oracle import edm_oracle as E
from oracle.denoiser_oracle import mask_pairs, mask_rows


def _toy_model(adj, node, flags, sig, sa, sn):
    """A cheap deterministic stand-in for the denoiser (the loop arithmetic is what is under test)."""
    return 0.9 * torch.tanh(adj * 0.3), 0.8 * torch.tanh(node * 0.2 + 0.1)


def _normal(seed):
    g = torch.Generator().manual_seed(seed)
    return lambda shape: torch.randn(shape, generator=g)


def _conditions(flags, c_e, c_n, seed, frac=0.5):
    """About `frac` of the valid nodes with class and box known, and every relation among the known nodes."""
    g = torch.Generator().manual_seed(seed)
    b, n = flags.shape
    nb = c_n - 4
    pick = flags & (torch.rand(b, n, generator=g) < frac)
    node_cls = torch.where(pick, torch.randint(0, 2 ** nb, (b, n), generator=g), torch.full((b, n), -1))
    bbox = torch.where(pick[..., None], torch.rand(b, n, 4, generator=g), torch.full((b, n, 4), float("nan")))
    pair = pick[:, :, None] & pick[:, None, :] & ~torch.eye(n, dtype=torch.bool)
    adj_cls = torch.where(pair, torch.randint(0, 2 ** c_e, (b, n, n), generator=g), torch.full((b, n, n), -1))
    return node_cls, bbox, adj_cls


def test_oracle_all_free_condition_is_the_plain_loop():
    cfg = CONFIGS["tiny"]
    flags = synthetic_node_flags(cfg, 3, seed=3)
    ce, cn = cfg["c_e"], cfg["c_n"]
    free = (torch.full((3, ce, 16, 16), float("nan")), torch.full((3, 16, cn), float("nan")))
    a0, n0 = E.sample(_toy_model, flags, ce, cn, num_steps=8, normal=_normal(4))
    a1, n1 = CO.sample(_toy_model, flags, ce, cn, free, num_steps=8, normal=_normal(4))
    assert torch.equal(a0, a1) and torch.equal(n0, n1)


def test_oracle_holds_known_entries_with_a_perfect_denoiser():
    cfg = CONFIGS["tiny"]
    ce, cn = cfg["c_e"], cfg["c_n"]
    flags = synthetic_node_flags(cfg, 3, seed=5)
    g = torch.Generator().manual_seed(6)
    gt = (mask_pairs(torch.randn(3, ce, 16, 16, generator=g).sign(), flags),
          mask_rows(torch.randn(3, 16, cn, generator=g).clamp(-1, 1), flags))
    known = CO.encode_known(flags, ce, cn, *_conditions(flags, ce, cn, seed=7))
    a, n = CO.sample(None, flags, ce, cn, known, num_steps=8, normal=_normal(8), gt=gt)
    ka, kn = ~known[0].isnan(), ~known[1].isnan()
    assert int(ka.sum()) > 0 and int(kn.sum()) > 0
    assert torch.equal(a[ka], known[0][ka]) and torch.equal(n[kn], known[1][kn])
    assert float((a - gt[0])[~ka].abs().max()) < 1e-6 and float((n - gt[1])[~kn].abs().max()) < 1e-6


@pytest.mark.parametrize("name", ["tiny", "vg", "coco"])
def test_oracle_encode_known_round_trips_through_decode(name):
    cfg = CONFIGS[name]
    ce, cn = cfg["c_e"], cfg["c_n"]
    flags = synthetic_node_flags(cfg, 4, seed=9)
    node_cls, bbox, adj_cls = _conditions(flags, ce, cn, seed=10, frac=1.0)
    ka, kn = CO.encode_known(flags, ce, cn, node_cls, bbox, adj_cls)
    qa, qn, box = E.decode_samples(ka.nan_to_num(0.0), kn.nan_to_num(0.0), flags, 2 ** ce, 2 ** (cn - 4))
    on_n = node_cls >= 0
    on_a = adj_cls >= 0
    assert torch.equal(qn.long()[on_n], node_cls[on_n]) and torch.equal(qa.long()[on_a], adj_cls[on_a])
    assert float((box[on_n] - bbox[on_n]).abs().max()) <= 1.2e-7
    # free entries stay NaN; class 0 ("no relation") is a constraint of its own: all bits -1
    assert bool(ka.permute(0, 2, 3, 1)[~on_a].isnan().all()) and bool(kn[~on_n].isnan().all())
    zero = adj_cls == 0
    if bool(zero.any()):
        assert bool((ka.permute(0, 2, 3, 1)[zero] == -1.0).all())


@pytest.fixture
def no_native(monkeypatch):
    """Every native entry point fails loudly: a ValueError must come first."""
    def boom(*a, **k):
        raise AssertionError("native code reached before the input checks")
    monkeypatch.setattr(native, "lib", boom)
    monkeypatch.setattr(native, "encode_known", boom)


def _base(b=2, n=8):
    flags = torch.zeros(b, n, dtype=torch.bool)
    flags[:, :5] = True
    return flags


@pytest.mark.parametrize("case", ["node_shape", "bbox_shape", "adj_shape", "node_range", "node_range_bits", "node_float",
                                  "adj_range", "adj_range_bits", "self_pair", "node_flag0", "bbox_flag0", "adj_flag0",
                                  "bbox_partial_nan", "bbox_inf", "bbox_range", "flags_shape", "types_too_many"])
def test_encode_known_rejects_bad_conditions_before_any_kernel(case, no_native):
    flags = _base()
    ce, cn = 3, 7            # 3 node class bits
    nc = torch.full((2, 8), -1)
    bb = torch.full((2, 8, 4), float("nan"))
    ac = torch.full((2, 8, 8), -1)
    kw = {}
    if case == "node_shape":
        nc = torch.full((2, 7), -1)
    elif case == "bbox_shape":
        bb = torch.zeros(2, 8, 3)
    elif case == "adj_shape":
        ac = torch.full((2, 8, 7), -1)
    elif case == "node_range":
        nc[0, 1] = 5
        kw = dict(num_node_type=5)
    elif case == "node_range_bits":
        nc[0, 1] = 8
    elif case == "node_float":
        nc = nc.float()
    elif case == "adj_range":
        ac[0, 1, 2] = 4
        kw = dict(num_adj_type=4)
    elif case == "adj_range_bits":
        ac[0, 1, 2] = -2
    elif case == "self_pair":
        ac[1, 3, 3] = 0
    elif case == "node_flag0":
        nc[1, 6] = 2
    elif case == "bbox_flag0":
        bb[0, 7] = 0.5
    elif case == "adj_flag0":
        ac[0, 2, 6] = 1
    elif case == "bbox_partial_nan":
        bb[0, 1] = torch.tensor([0.1, float("nan"), 0.3, 0.4])
    elif case == "bbox_inf":
        bb[0, 1] = torch.tensor([0.1, float("inf"), 0.3, 0.4])
    elif case == "bbox_range":
        bb[0, 1] = torch.tensor([0.1, 0.2, 1.5, 0.4])
    elif case == "flags_shape":
        flags = flags[0]
    elif case == "types_too_many":
        kw = dict(num_node_type=9)
    with pytest.raises(ValueError):
        completion.encode_known(flags, ce, cn, node_cls=nc, bbox=bb, adj_cls=ac, **kw)


def _sampler():
    return NodeAdjEDMSampler(num_steps=4, clip_samples=True, clip_samples_min=-1.0, clip_samples_max=1.0,
                             clip_samples_scope="x_0", dev="cpu", objective="edm", self_condition=True,
                             symmetric_noise=False)


@pytest.mark.parametrize("case", ["adj_shape", "node_shape", "adj_outside_pair", "node_outside_flags", "inf",
                                  "int_dtype"])
def test_sample_completion_rejects_bad_conditions_before_any_kernel(case, no_native):
    flags = _base()
    ka = torch.full((2, 3, 8, 8), float("nan"))
    kn = torch.full((2, 8, 7), float("nan"))
    if case == "adj_shape":
        ka = ka[:, :2]
    elif case == "node_shape":
        kn = kn[..., :6]
    elif case == "adj_outside_pair":
        ka[1, 0, 2, 6] = 1.0
    elif case == "node_outside_flags":
        kn[0, 5, 0] = -1.0
    elif case == "inf":
        ka[0, 0, 1, 2] = float("-inf")
    elif case == "int_dtype":
        ka = torch.zeros(2, 3, 8, 8, dtype=torch.int32)
    with pytest.raises(ValueError):
        _sampler().sample_completion(None, flags, ka, kn, num_node_chan=7, num_edge_chan=3)


def test_known_answer_mode_cannot_be_combined_with_known_entries(no_native):
    flags = _base()
    known = (torch.full((2, 3, 8, 8), float("nan")), torch.full((2, 8, 7), float("nan")))
    gt = (torch.zeros(2, 3, 8, 8), torch.zeros(2, 8, 7))
    with pytest.raises(ValueError):
        _sampler()._sample_on_device(None, flags, sanity_check_gt_adjs=gt[0], sanity_check_gt_nodes=gt[1],
                                     num_node_chan=7, num_edge_chan=3, known=known)


def test_valid_conditions_pass_the_checks():
    flags = _base()
    nc = torch.full((2, 8), -1)
    nc[0, :3] = torch.tensor([0, 7, 3])
    bb = torch.full((2, 8, 4), float("nan"))
    bb[1, 4] = torch.tensor([0.0, 1.0, 0.25, 0.5])
    ac = torch.full((2, 8, 8), -1)
    ac[0, 0, 1] = 0
    ac[1, 4, 2] = 7
    completion.validate_conditions(flags, 3, 7, nc, bb, ac)
    completion.validate_conditions(flags, 3, 7, nc, bb, ac, num_adj_type=8, num_node_type=8)
    completion.validate_conditions(flags, 3, 7)
