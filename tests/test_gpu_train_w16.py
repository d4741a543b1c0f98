"""Training the 16 x 16-window geometry (n64w16, T = 256 tokens per window) on the B200 (run with -m gpu): the window-
attention backward dsg_tr_window_attention_bwd_w16 against torch autograd on the GPU, the whole denoiser's parameter
gradients against torch autograd of the CPU oracle, the graphed training step against the eager one, and the refusal of
non-reference index / mask buffers."""
import numpy as np
import pytest
import torch

from diffusesg_b200 import native
from diffusesg_b200.loss.rainbow_loss import NodeAdjRainbowLoss
from diffusesg_b200.model.diffusesg.diffusesg import DiffuseSG
from diffusesg_b200.model.diffusesg.geometry import relative_position_index, shifted_window_mask
from diffusesg_b200.model.diffusesg.train_graph import train_state
from diffusesg_b200.model.precond.precond import NodeAdjPrecond
from diffusesg_b200.runner.objectives.edm import NodeAdjEDMObjectiveGenerator
from diffusesg_b200.runner.trainer.trainer_node_adj import train_one_step
from diffusesg_b200.utils.synthetic import CONFIGS, in_chans, synthetic_inputs, synthetic_state_dict
from diffusesg_b200.utils.train_utils import FusedAdam, GraphedTrainStep, NativeEMA
from oracle import denoiser_oracle as O

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CFG = CONFIGS["n64w16"]


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


# ---------------------------------------------------------------------------------------------------------
# the kernel
# ---------------------------------------------------------------------------------------------------------
def _attention_reference(qkv, bias, mask, batch, res, w, shift, heads):
    """WindowAttention.forward with roll / window_partition / window_reverse, fp32 (as in test_gpu_train.py)."""
    c = heads * 32
    x = qkv.view(batch, res, res, 3 * c)
    if shift:
        x = torch.roll(x, shifts=(-shift, -shift), dims=(1, 2))
    nw = res // w
    t = w * w
    xw = x.view(batch, nw, w, nw, w, 3 * c).permute(0, 1, 3, 2, 4, 5).reshape(batch * nw * nw, t, 3, heads, 32)
    q, k, v = xw.permute(2, 0, 3, 1, 4)
    att = q @ k.transpose(-1, -2) + bias[None]
    if mask is not None:
        att = (att.view(batch, nw * nw, heads, t, t) + mask[None, :, None]).view(-1, heads, t, t)
    out = (att.softmax(-1) @ v).transpose(1, 2).reshape(batch, nw, nw, w, w, c).permute(0, 1, 3, 2, 4, 5)
    out = out.reshape(batch, res, res, c)
    if shift:
        out = torch.roll(out, shifts=(shift, shift), dims=(1, 2))
    return out.reshape(batch * res * res, c)


def _inputs(batch, res, shift, heads):
    g = torch.Generator(device=DEV).manual_seed(res * 100 + shift + heads + batch)
    c = heads * 32
    qkv = torch.randn(batch * res * res, 3 * c, device=DEV, generator=g)
    qkv[:, :c] *= 32 ** -0.5
    datt = torch.randn(batch * res * res, c, device=DEV, generator=g)
    table = torch.randn(31 * 31, heads, device=DEV, generator=g) * 0.5
    return qkv.to(torch.bfloat16), datt.to(torch.bfloat16), table


def _backward_w16(qkv, datt, table, batch, res, shift, heads):
    dqkv = torch.empty_like(qkv)
    dtable = torch.zeros_like(table)
    native.check(native.lib().dsg_tr_window_attention_bwd_w16(qkv.data_ptr(), datt.data_ptr(), table.data_ptr(),
                                                              dqkv.data_ptr(), dtable.data_ptr(), batch, res, 16, shift,
                                                              heads, native.stream_ptr(DEV)), "attention_bwd_w16")
    torch.cuda.synchronize()
    return dqkv, dtable


@pytest.mark.parametrize("batch,res,shift,heads", [(2, 16, 0, 12), (3, 32, 8, 6), (2, 64, 0, 3), (2, 64, 8, 3), (5, 32, 0, 6),
                                                   (40, 64, 8, 3)])
def test_window_attention_backward_w16(batch, res, shift, heads):
    """Against autograd of the fp32 attention with the reference's relative_position_index and SW-MSA mask; (40, 64, 8, 3)
    gives every CTA many items before its table flush."""
    qkv, datt, table = _inputs(batch, res, shift, heads)
    index = relative_position_index(16).to(DEV)
    mask = shifted_window_mask(res, 16, shift).to(DEV) if shift else None
    q32 = qkv.float().requires_grad_(True)
    tab = table.clone().requires_grad_(True)
    bias_ref = tab[index.reshape(-1)].view(256, 256, heads).permute(2, 0, 1)
    (_attention_reference(q32, bias_ref, mask, batch, res, 16, shift, heads) * datt.float()).sum().backward()
    dqkv, dtable = _backward_w16(qkv, datt, table, batch, res, shift, heads)
    # the bounds of test_window_attention_backward: bf16 operands of the tensor-core products (P and dS rounded like the
    # forward's P) and of the stored gradient; the table gradient sums the fp32 dS
    e_qkv, e_tab = _rel(dqkv.float(), q32.grad), _rel(dtable, tab.grad)
    print(f"dqkv rel-L2 {e_qkv:.2e}, dtable rel-L2 {e_tab:.2e}")
    assert e_qkv < 1e-2, e_qkv
    assert e_tab < 2e-3, e_tab
    again, _ = _backward_w16(qkv, datt, table, batch, res, shift, heads)
    assert torch.equal(again, dqkv)      # every element written once, no atomics: bit-identical


def test_window_attention_backward_w16_ignores_shared_memory_leftovers():
    """All shared memory overwritten with NaN after every launch: dqkv is bit-identical, the table gradient agrees up to the
    order of its atomic per-CTA flushes."""
    shape = (3, 32, 8, 6)
    qkv, datt, table = _inputs(*shape)
    out = []
    for poison in (0, 1):
        native.lib().dsg_debug_set_smem_poison(0x7fc00000, poison)
        try:
            _backward_w16(qkv, datt, table, *shape)     # leaves the poison behind for the next launch
            out.append(_backward_w16(qkv, datt, table, *shape))
        finally:
            native.lib().dsg_debug_set_smem_poison(0, 0)
    (d0, t0), (d1, t1) = out
    assert torch.equal(d0, d1)
    assert torch.isfinite(t1).all() and _rel(t1, t0) < 1e-5, _rel(t1, t0)


# ---------------------------------------------------------------------------------------------------------
# the whole denoiser
# ---------------------------------------------------------------------------------------------------------
def _net(sd):
    net = DiffuseSG(img_size=CFG["img"], in_chans=in_chans(CFG), patch_size=1, embed_dim=CFG["embed"], depths=CFG["depths"],
                    num_heads=[3, 6, 12, 24], window_size=CFG["window"], mlp_ratio=4., drop_rate=0., attn_drop_rate=0.,
                    drop_path_rate=0.0, self_condition=True, symmetric_noise=False, out_chans_adj=CFG["c_e"],
                    out_chans_node=CFG["c_n"])
    net.load_state_dict(sd, strict=True)
    return net.to(DEV)


def test_denoiser_parameter_gradients_match_oracle_autograd_n64w16():
    """Method of test_gpu_train.py::test_denoiser_parameter_gradients_match_oracle_autograd on the 16 x 16-window geometry:
    three stages with 16 x 16 windows (res 64 and 32 shifted every other block, res 16 one window) and one with 8 x 8."""
    batch = 2
    sd = synthetic_state_dict(CFG, seed=1234, stress=True)
    adj, node, flags, _, sc_adj, sc_node = synthetic_inputs(CFG, batch, seed=11)
    sigmas = torch.tensor([0.2, 1.5])       # one noise level per sample, as in training
    g = torch.Generator().manual_seed(5)
    wa, wn = torch.randn(adj.shape, generator=g), torch.randn(node.shape, generator=g)
    leaves = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "attn_mask" not in k else v) for k, v in sd.items()}

    def onet(a, x, f, c_noise, sa, sn):
        return O.denoiser_forward(leaves, img=CFG["img"], embed=CFG["embed"], depths=CFG["depths"], heads=CFG["heads"],
                                  window=CFG["window"], self_condition=True, adj=a, node=x, flags=f, noise_labels=c_noise,
                                  sc_adj=sa, sc_node=sn)
    ref_a, ref_n = O.precond_forward(onet, adj, node, flags, sigmas, sc_adj, sc_node)
    ((ref_a * wa).sum() + (ref_n * wn).sum()).backward()
    ref_g = {k: v.grad for k, v in leaves.items() if v.is_floating_point() and v.requires_grad}
    net = _net(sd).train()
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=False, symmetric_noise=False).train()
    da, dn = model(adj.to(DEV), node.to(DEV), flags.to(DEV), sigmas.to(DEV), sc_adj.to(DEV), sc_node.to(DEV))
    ea, en = _rel(da.detach().cpu(), ref_a.detach()), _rel(dn.detach().cpu(), ref_n.detach())
    assert ea < 2.5e-2 and en < 2.5e-2, (ea, en)
    ((da * wa.to(DEV)).sum() + (dn * wn.to(DEV)).sum()).backward()
    torch.cuda.synchronize()
    params = dict(net.named_parameters())
    worst, num, den = [], 0.0, 0.0
    for k, gr in ref_g.items():
        if gr is None:
            continue
        got = params[k].grad
        assert got is not None and torch.isfinite(got).all(), k
        d = got.detach().cpu().double() - gr.double()
        num += float(d.pow(2).sum())
        den += float(gr.double().pow(2).sum())
        worst.append((float(d.norm() / gr.double().norm().clamp_min(1e-30)), k, float(gr.norm())))
    worst.sort(reverse=True)
    total = (num / den) ** 0.5
    print(f"n64w16: outputs {ea:.2e} / {en:.2e}; all-parameter gradient rel-L2 {total:.3e}; worst " +
          ", ".join(f"{k} {e:.2e}" for e, k, _ in worst[:5]))
    # the all-parameter bound of the shallower geometries (4e-2) does not hold here, and not because of the attention
    # backward: the error comes from the bf16 operands of the GEMMs, compounded through 24 blocks instead of 12.  Measured
    # on a B200: 5.04e-2 with dsg_tr_window_attention_bwd_w16, 5.09e-2 with an exact fp32 attention backward in its place;
    # the reference's OWN bf16-autocast gradients (torch CPU autocast of the oracle, same inputs) sit 9.1e-2 from its fp32
    # ones on this geometry (4.5e-2 on VG).  The per-tensor bound below is unchanged.
    assert total < 6e-2, (total, worst[:8])
    gmax = max(n for _, _, n in worst)
    for e, k, n in worst:
        if n > 1e-3 * gmax:
            assert e < 1e-1, (k, e)


def test_graphed_training_step_matches_eager_n64w16():
    """test_gpu_train.py::test_graphed_training_step_matches_eager on the 16 x 16-window geometry, same bounds."""
    adj, node, flags, *_ = synthetic_inputs(CFG, 4, seed=3)
    adj, node = O.mask_pairs(adj.sign(), flags).to(DEV), O.mask_rows(node.clamp(-1, 1), flags).to(DEV)
    flags = flags.to(DEV)
    runs = []
    for graphed in (False, True):
        net = _net(synthetic_state_dict(CFG, seed=1234, stress=False)).train()
        model = NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).train()
        opt = FusedAdam(model, lr=1e-3, max_grad_norm=10.0)
        emas = [NativeEMA(model, beta=0.99)]
        opt.attach_emas(emas)
        gen = NodeAdjEDMObjectiveGenerator("edm", "edm", dev=DEV, symmetric_noise=False)
        loss_fn = NodeAdjRainbowLoss(edge_loss_weight=1.0, node_loss_weight=1.0, objective="edm")
        step = GraphedTrainStep(model, opt, emas, gen, loss_fn) if graphed else None
        np.random.seed(4)
        losses = []
        for it in range(8):
            torch.manual_seed(50 + it)
            if graphed:
                la, ln = step(adj, node, flags)
            else:
                la, ln = train_one_step(model, opt, emas, gen, loss_fn, adj, node, flags)
            losses.append(float(la.mean() + ln.mean()))
        torch.cuda.synchronize()
        runs.append((losses, train_state(net, DEV).flat.clone(), emas[0].flat.clone(), model.raw_passes))
    (l0, w0, e0, p0), (l1, w1, e1, p1) = runs
    assert p0 == p1 and 8 < p0 < 16                       # both coin outcomes were exercised
    assert all(np.isfinite(l0)) and np.allclose(l0, l1, rtol=2e-3), (l0, l1)
    assert _rel(w1, w0) < 5e-3 and _rel(e1, e0) < 5e-3, (_rel(w1, w0), _rel(e1, e0))


# ---------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("what", ["relative_position_index", "attn_mask"])
def test_backward_refuses_non_reference_w16_buffers(what):
    """The forward runs with any buffers (the generic attention kernel takes them); the backward of a 16 x 16 block needs
    the reference's and raises before any kernel of that block runs."""
    prefix = "up_layers.3.blocks.1"      # 64 x 64 tokens, shift 8: the first block the backward reaches
    net = _net(synthetic_state_dict(CFG, seed=1234, stress=False)).train()
    blk = net.get_submodule(prefix)
    with torch.no_grad():
        if what == "relative_position_index":
            idx = blk.attn.relative_position_index
            idx[0, 1], idx[0, 2] = idx[0, 2].clone(), idx[0, 1].clone()
        else:
            blk.attn_mask[0, 0, 1] = -100.0    # window 0 lies in one region: the reference's mask is 0 there
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=False, symmetric_noise=False).train()
    adj, node, flags, sigmas, _, _ = [t.to(DEV) for t in synthetic_inputs(CFG, 2, seed=11)]
    da, dn = model(adj, node, flags, sigmas)
    with pytest.raises(NotImplementedError, match=f"{prefix}.{'attn.' if what != 'attn_mask' else ''}{what}"):
        (da.square().mean() + dn.square().mean()).backward()
    torch.cuda.synchronize()
    st = train_state(net, DEV)
    assert float(st.g(prefix + ".mlp.fc2.weight").abs().sum()) == 0.0
    assert float(st.g(prefix + ".attn.relative_position_bias_table").abs().sum()) == 0.0
