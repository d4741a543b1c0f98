"""Input gradients and guided completion without a GPU: the new entry points reject bad arguments before they touch a
pointer or the device, sample_completion rejects a bad guidance scale before any kernel, and the completion oracle's
reconstruction guidance (oracle/guided_completion_oracle.py, DESIGN.md §3.7) against a closed form and against the unguided loop."""
import pytest
import torch

from diffusesg_b200 import native
from diffusesg_b200.runner.mcmc_sampler.edm import NodeAdjEDMSampler
from diffusesg_b200.utils.synthetic import CONFIGS, synthetic_node_flags
from oracle import completion_oracle as CO
from oracle import guided_completion_oracle as GO
from oracle import edm_oracle as E
from oracle.denoiser_oracle import mask_pairs, mask_rows

DSG_ERR_INVALID = 1
FAKE = 4096        # a 16-byte aligned address that is never dereferenced: the arguments are checked first


# ---------------------------------------------------------------------------------------------------------
# C ABI argument checks
# ---------------------------------------------------------------------------------------------------------
def _embed_bwd(**kw):
    a = dict(dinp=FAKE, g_adj=FAKE, g_node=FAKE, flags=FAKE, c_in=FAKE, c_skip=FAKE, d_adj=FAKE, d_node=FAKE, B=2, n=16,
             c_e=3, c_n=5, self_cond=1, ld=96)
    a.update(kw)
    return native.lib().dsg_tr_embed_input_bwd(a["dinp"], a["g_adj"], a["g_node"], a["flags"], a["c_in"], a["c_skip"],
                                               a["d_adj"], a["d_node"], a["B"], a["n"], a["c_e"], a["c_n"],
                                               a["self_cond"], a["ld"], None)


@pytest.mark.parametrize("case", [
    dict(dinp=None), dict(flags=None), dict(d_adj=None), dict(d_node=None),
    dict(c_in=None), dict(c_skip=None), dict(g_adj=None), dict(g_node=None),
    dict(ld=92), dict(ld=20), dict(c_e=40, ld=96), dict(self_cond=1, c_e=20, c_n=8, ld=64), dict(dinp=FAKE + 4),
    dict(B=0), dict(n=0), dict(c_e=0), dict(c_n=0), dict(B=70000), dict(ld=256, c_n=5, c_e=3)])
def test_embed_input_bwd_rejects_bad_arguments(case):
    assert _embed_bwd(**case) == DSG_ERR_INVALID
    assert native.lib().dsg_last_error().decode().startswith("tr_embed_input_bwd")


def test_embed_input_bwd_raw_mode_needs_no_output_gradients():
    # c_in == c_skip == NULL (raw F): the output gradients are not read, so they may be NULL; ld % 8 is still checked
    assert _embed_bwd(c_in=None, c_skip=None, g_adj=None, g_node=None, ld=90) == DSG_ERR_INVALID
    assert "ld % 8" in native.lib().dsg_last_error().decode()


def _residual(**kw):
    a = dict(d_adj=FAKE, d_node=FAKE, k_adj=FAKE, k_node=FAKE, flags=FAKE, r_adj=FAKE, r_node=FAKE, b=2, ce=3, n=16, cn=5)
    a.update(kw)
    return native.lib().dsg_edm_guidance_residual(a["d_adj"], a["d_node"], a["k_adj"], a["k_node"], a["flags"], a["r_adj"],
                                                  a["r_node"], a["b"], a["ce"], a["n"], a["cn"], None)


def _update(**kw):
    a = dict(d_adj=FAKE, d_node=FAKE, g_adj=FAKE, g_node=FAKE, flags=FAKE, w=1.0, o_adj=FAKE, o_node=FAKE, b=2, ce=3, n=16,
             cn=5)
    a.update(kw)
    return native.lib().dsg_edm_guidance_update(a["d_adj"], a["d_node"], a["g_adj"], a["g_node"], a["flags"], a["w"],
                                                a["o_adj"], a["o_node"], a["b"], a["ce"], a["n"], a["cn"], None)


@pytest.mark.parametrize("case", [dict(d_adj=None), dict(k_node=None), dict(flags=None), dict(r_adj=None), dict(n=18),
                                  dict(b=0), dict(d_adj=FAKE + 4), dict(flags=FAKE + 1)])
def test_guidance_residual_rejects_bad_arguments(case):
    assert _residual(**case) == DSG_ERR_INVALID


@pytest.mark.parametrize("case", [dict(g_adj=None), dict(o_node=None), dict(w=-0.5), dict(w=float("nan")),
                                  dict(w=float("inf")), dict(n=10), dict(cn=0), dict(o_adj=FAKE + 8)])
def test_guidance_update_rejects_bad_arguments(case):
    assert _update(**case) == DSG_ERR_INVALID


# ---------------------------------------------------------------------------------------------------------
# sample_completion: the guidance scale is checked before anything runs
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture
def no_native(monkeypatch):
    def boom(*a, **k):
        raise AssertionError("native code reached before the input checks")
    monkeypatch.setattr(native, "lib", boom)


@pytest.mark.parametrize("w", [-1e-3, float("nan"), float("inf"), -float("inf")])
def test_sample_completion_rejects_bad_guidance_scale(w, no_native):
    flags = torch.zeros(2, 8, dtype=torch.bool)
    flags[:, :5] = True
    ka = torch.full((2, 3, 8, 8), float("nan"))
    kn = torch.full((2, 8, 7), float("nan"))
    s = NodeAdjEDMSampler(num_steps=4, clip_samples=True, clip_samples_min=-1.0, clip_samples_max=1.0,
                          clip_samples_scope="x_0", dev="cpu", objective="edm", self_condition=True, symmetric_noise=False)
    with pytest.raises(ValueError, match="guidance_scale"):
        s.sample_completion(None, flags, ka, kn, num_node_chan=7, num_edge_chan=3, guidance_scale=w)


# ---------------------------------------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------------------------------------
def _toy_model(adj, node, flags, sig, sa, sn):
    """A cheap differentiable stand-in for the denoiser: D = (0.9 tanh(0.3 adj), 0.8 tanh(0.2 node + 0.1))."""
    return 0.9 * torch.tanh(adj * 0.3), 0.8 * torch.tanh(node * 0.2 + 0.1)


def _normal(seed):
    g = torch.Generator().manual_seed(seed)
    return lambda shape: torch.randn(shape, generator=g)


def _known(flags, ce, cn, seed, frac=0.5):
    g = torch.Generator().manual_seed(seed)
    b, n = flags.shape
    pair = (flags[:, :, None] & flags[:, None, :])[:, None].expand(b, ce, n, n)
    ka = torch.where(pair & (torch.rand(b, ce, n, n, generator=g) < frac), torch.randn(b, ce, n, n, generator=g).sign(),
                     float("nan"))
    kn = torch.where(flags[..., None] & (torch.rand(b, n, cn, generator=g) < frac),
                     torch.rand(b, n, cn, generator=g) * 2 - 1, float("nan"))
    return ka, kn


def _setup():
    cfg = CONFIGS["tiny"]
    flags = synthetic_node_flags(cfg, 3, seed=3)
    return cfg["c_e"], cfg["c_n"], flags, _known(flags, cfg["c_e"], cfg["c_n"], 9)


def test_oracle_zero_guidance_is_the_completion_loop():
    ce, cn, flags, known = _setup()
    a0, n0 = CO.sample(_toy_model, flags, ce, cn, known, num_steps=8, normal=_normal(4))
    a1, n1 = GO.sample(_toy_model, flags, ce, cn, known, num_steps=8, normal=_normal(4), guidance=0.0)
    assert torch.equal(a0, a1) and torch.equal(n0, n1)


def test_oracle_guidance_without_known_entries_is_the_plain_loop():
    ce, cn, flags, _ = _setup()
    free = (torch.full((3, ce, 16, 16), float("nan")), torch.full((3, 16, cn), float("nan")))
    a0, n0 = E.sample(_toy_model, flags, ce, cn, num_steps=8, normal=_normal(4))
    a1, n1 = GO.sample(_toy_model, flags, ce, cn, free, num_steps=8, normal=_normal(4), guidance=0.7)
    assert torch.equal(a0, a1) and torch.equal(n0, n1)


def test_oracle_guided_denoiser_matches_closed_form():
    """For the elementwise toy denoiser the guidance gradient is r * D'(x) on the known entries."""
    ce, cn, flags, known = _setup()
    g = torch.Generator().manual_seed(2)
    xa = mask_pairs(torch.randn(3, ce, 16, 16, generator=g) * 3, flags)
    xn = mask_rows(torch.randn(3, 16, cn, generator=g) * 3, flags)
    w = 0.6
    got_a, got_n = GO.guided(_toy_model, xa, xn, flags, None, None, None, known, w)
    da, dn = _toy_model(xa, xn, flags, None, None, None)
    da, dn = mask_pairs(da, flags), mask_rows(dn, flags)
    ra = torch.where(known[0].isnan(), 0.0, da - torch.nan_to_num(known[0]))
    rn = torch.where(known[1].isnan(), 0.0, dn - torch.nan_to_num(known[1]))
    ga = mask_pairs(ra * 0.27 * (1 - torch.tanh(0.3 * xa) ** 2), flags)
    gn = mask_rows(rn * 0.16 * (1 - torch.tanh(0.2 * xn + 0.1) ** 2), flags)
    torch.testing.assert_close(got_a, mask_pairs(da - w * ga, flags), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(got_n, mask_rows(dn - w * gn, flags), rtol=1e-6, atol=1e-6)


def _coupled_model(adj, node, flags, sig, sa, sn):
    """Toy denoiser whose outputs depend on other entries (an elementwise one leaves the free entries unguided)."""
    return (0.9 * torch.tanh(adj * 0.3 + 0.5 * adj.mean((1, 2, 3), keepdim=True)),
            0.8 * torch.tanh(node * 0.2 + 0.5 * node.mean((1, 2), keepdim=True)))


def test_oracle_guidance_changes_the_sample_and_holds_known_entries():
    ce, cn, flags, known = _setup()
    a0, n0 = CO.sample(_coupled_model, flags, ce, cn, known, num_steps=8, normal=_normal(4))
    a1, n1 = GO.sample(_coupled_model, flags, ce, cn, known, num_steps=8, normal=_normal(4), guidance=1.0)
    fa, fn = ~known[0].isnan(), ~known[1].isnan()
    assert torch.equal(a1[fa], known[0][fa]) and torch.equal(n1[fn], known[1][fn])
    pair = (flags[:, None, :, None] & flags[:, None, None, :]).expand_as(a0)
    assert not torch.equal(a0[~fa & pair], a1[~fa & pair])
    assert float(a1[~pair].abs().sum()) == 0.0 and float(n1[~flags].abs().sum()) == 0.0
