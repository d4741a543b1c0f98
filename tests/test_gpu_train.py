"""Training step on the B200 (SURVEY 8 f-2; run with -m gpu): every backward kernel against torch autograd of the same
op on the GPU, and the whole denoiser's parameter gradients against torch autograd of the CPU oracle
(oracle/denoiser_oracle.py, fp32) on the same weights and inputs.  Everything goes through the C ABI."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from diffusesg_b200 import native
from diffusesg_b200.loss.rainbow_loss import NodeAdjRainbowLoss
from diffusesg_b200.model.diffusesg.diffusesg import DiffuseSG
from diffusesg_b200.model.diffusesg.geometry import relative_position_index, shifted_window_mask
from diffusesg_b200.model.diffusesg.train_graph import _Ops, train_state
from diffusesg_b200.model.precond.precond import NodeAdjPrecond
from diffusesg_b200.runner.objectives.edm import NodeAdjEDMObjectiveGenerator
from diffusesg_b200.runner.trainer.trainer_node_adj import train_one_step
from diffusesg_b200.utils.synthetic import CONFIGS, in_chans, synthetic_inputs, synthetic_state_dict
from diffusesg_b200.utils.train_utils import FusedAdam, GraphedTrainStep, NativeEMA
from oracle import denoiser_oracle as O
from oracle import train_oracle as T

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def _ops():
    return _Ops(DEV)


# ---------------------------------------------------------------------------------------------------------
# row kernels
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,Cdim", [(777, 96), (1000, 384), (130, 1536), (4096, 192)])
def test_layernorm_forward_backward(M, Cdim):
    g = torch.Generator(device=DEV).manual_seed(M + Cdim)
    x = (torch.randn(M, Cdim, device=DEV, generator=g) * 2 + 0.5).requires_grad_(True)
    gamma = (1 + 0.2 * torch.randn(Cdim, device=DEV, generator=g)).requires_grad_(True)
    beta = (0.1 * torch.randn(Cdim, device=DEV, generator=g)).requires_grad_(True)
    dy = torch.randn(M, Cdim, device=DEV, generator=g)
    extra = torch.randn(M, Cdim, device=DEV, generator=g)
    want = F.layer_norm(x, (Cdim,), gamma, beta, 1e-5)
    (want * dy).sum().backward()
    o = _ops()
    y16, y32 = o.ln_fwd(x.detach(), gamma.detach(), beta.detach(), bf16=True, f32=True)
    assert _rel(y32, want) < 2e-6 and _rel(y16.float(), want) < 4e-3
    dgamma, dbeta = torch.zeros(Cdim, device=DEV), torch.zeros(Cdim, device=DEV)
    dx = o.ln_bwd(dy, x.detach(), gamma.detach(), dgamma, dbeta, dx_add=extra.clone())
    assert _rel(dx, x.grad + extra) < 1e-5
    assert _rel(dgamma, gamma.grad) < 1e-4 and _rel(dbeta, beta.grad) < 1e-4


@pytest.mark.parametrize("B,L,Cdim", [(3, 100, 96), (2, 4096, 96), (5, 64, 768)])
def test_film_silu_forward_backward(B, L, Cdim):
    g = torch.Generator(device=DEV).manual_seed(B + L)
    ld, off = 2 * Cdim + 64, 32
    v = torch.randn(B * L, Cdim, device=DEV, generator=g).requires_grad_(True)
    film = (0.5 * torch.randn(B, ld, device=DEV, generator=g)).requires_grad_(True)
    dout = torch.randn(B * L, Cdim, device=DEV, generator=g)
    sc, sh = film[:, off:off + Cdim], film[:, off + Cdim:off + 2 * Cdim]
    want = F.silu(torch.addcmul(sh[:, None], v.view(B, L, Cdim), sc[:, None] + 1)).reshape(B * L, Cdim)
    (want * dout).sum().backward()
    o = _ops()
    got = o.film_fwd(v.detach(), film.detach(), off, B, L, Cdim)
    assert _rel(got, want) < 2e-6
    dfilm = torch.zeros(B, ld, device=DEV)
    dv = o.film_bwd(dout, v.detach(), film.detach(), off, dfilm, B, L, Cdim)
    assert _rel(dv, v.grad) < 1e-5 and _rel(dfilm, film.grad) < 1e-4


def test_gelu_and_silu():
    g = torch.Generator(device=DEV).manual_seed(1)
    pre = (torch.randn(1000, 384, device=DEV, generator=g) * 2).to(torch.bfloat16)
    dh = torch.randn(1000, 384, device=DEV, generator=g).to(torch.bfloat16)
    p32 = pre.float().requires_grad_(True)
    want = F.gelu(p32)
    (want * dh.float()).sum().backward()
    o = _ops()
    assert _rel(o.gelu(pre).float(), want) < 4e-3
    assert _rel(o.gelu(pre, dh).float(), p32.grad) < 4e-3
    x = torch.randn(50, 512, device=DEV, generator=g).requires_grad_(True)
    d = torch.randn(50, 512, device=DEV, generator=g)
    (F.silu(x) * d).sum().backward()
    assert _rel(o.silu(x.detach()), F.silu(x)) < 1e-6 and _rel(o.silu(x.detach(), d), x.grad) < 1e-5
    y = torch.randn(70, 96, device=DEV, generator=g).requires_grad_(True)
    (F.gelu(y) * d[:, :96].repeat(2, 1)[:70]).sum().backward()
    assert _rel(o.gelu_f32(y.detach()), F.gelu(y)) < 1e-6
    assert _rel(o.gelu_f32(y.detach(), d[:, :96].repeat(2, 1)[:70].contiguous()), y.grad) < 1e-5


def test_shuffle_and_copy_cols():
    B, H, W, Cdim = 3, 4, 6, 8
    fine = torch.randn(B, 2 * H, 2 * W, Cdim, device=DEV)
    want = torch.cat([fine[:, 0::2, 0::2], fine[:, 1::2, 0::2], fine[:, 0::2, 1::2], fine[:, 1::2, 1::2]], -1)  # :325-329
    o = _ops()
    coarse = o.shuffle(fine.reshape(-1, Cdim), B, H, W, Cdim, True)
    assert torch.equal(coarse.view(B, H, W, 4 * Cdim), want)
    back = o.shuffle(coarse, B, H, W, Cdim, False)
    assert torch.equal(back.view_as(fine), fine)
    x = torch.randn(100, 16, device=DEV)
    cat = torch.zeros(100, 40, device=DEV, dtype=torch.bfloat16)
    o.copy_cols(x, 4, cat, 24, 12)
    assert torch.equal(cat[:, 24:36].float(), x[:, 4:16].to(torch.bfloat16).float()) and float(cat[:, :24].abs().sum()) == 0
    acc = torch.ones(100, 16, device=DEV)
    o.copy_cols(x, 0, acc, 0, 16, accumulate=True)
    assert torch.allclose(acc, x + 1)


# ---------------------------------------------------------------------------------------------------------
# GEMMs of the backward pass
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_out,x_cols,out_cols,M,scale_rows", [
    (96, 96, 96, 4096, 0), (288, 96, 96, 20000, 96), (384, 1536, 1536, 8192, 0), (1536, 384, 384, 3008, 0),
    (96, 96, 60, 5008, 0), (768, 768, 768, 48, 0), (2304, 768, 768, 1024, 768), (96, 384, 384, 524288, 0), (192, 192, 192, 64, 0)])
def test_weight_gradient_mn_major(n_out, x_cols, out_cols, M, scale_rows):
    """dW += dY^T X on the tcgen05 kernel with MN-major operands (dY and X read as they lie, no transposes), split-K."""
    g = torch.Generator(device=DEV).manual_seed(n_out + M)
    dy = torch.randn(M, n_out, device=DEV, generator=g).to(torch.bfloat16)
    x = torch.randn(M, x_cols, device=DEV, generator=g).to(torch.bfloat16)
    if out_cols != x_cols:
        x[:, out_cols:] = 0
    o = _ops()
    dw = torch.full((n_out, out_cols), 0.5, device=DEV)
    o.wgrad_mn(dy, x, dw, scale_rows=scale_rows, scale=0.25)
    torch.cuda.synchronize()
    want = dy.float().t() @ x.float()[:, :out_cols]
    want[:scale_rows] *= 0.25
    want += 0.5
    assert _rel(dw, want) < 2e-5, _rel(dw, want)


@pytest.mark.parametrize("M,Cdim,bf16", [(1000, 96, False), (2056, 288, True), (50, 1536, False), (70000, 384, True)])
def test_cast_colsum(M, Cdim, bf16):
    g = torch.Generator(device=DEV).manual_seed(M)
    src = torch.randn(M, Cdim, device=DEV, generator=g)
    if bf16:
        src = src.to(torch.bfloat16)
    colsum = torch.ones(Cdim, device=DEV)
    o = _ops()
    cast = o.cast_colsum(src, colsum=colsum, cast=not bf16, scale_cols=40, scale=0.25)
    ref = src.float().sum(0)
    ref[:40] *= 0.25
    assert _rel(colsum - 1, ref) < 1e-4
    if not bf16:
        assert torch.equal(cast.float(), src.to(torch.bfloat16).float())


@pytest.mark.parametrize("M,N,K", [(128, 512, 96), (100, 9000, 512), (8192, 12, 96), (70000, 6, 96)])
def test_small_fp32_gemm(M, N, K):
    g = torch.Generator(device=DEV).manual_seed(M + N)
    x = torch.randn(M, K, device=DEV, generator=g)
    w = torch.randn(N, K, device=DEV, generator=g) / K ** 0.5
    b = torch.randn(N, device=DEV, generator=g)
    dy = torch.randn(M, N, device=DEV, generator=g)
    o = _ops()
    assert _rel(o.linear_small(x, w, b), x @ w.t() + b) < 1e-5
    dw, db = torch.zeros(N, K, device=DEV), torch.zeros(N, device=DEV)
    dx = o.linear_small_bwd(dy, x, w, dw, db)
    assert _rel(dx, dy @ w) < 1e-5 and _rel(dw, dy.t() @ x) < 1e-4 and _rel(db, dy.sum(0)) < 1e-4
    xb = x.to(torch.bfloat16)
    dw2 = torch.zeros(N, K, device=DEV)
    o.linear_small_bwd(dy, xb, w, dw2, None, need_dx=False)
    assert _rel(dw2, dy.t() @ xb.float()) < 1e-4


@pytest.mark.parametrize("M,E,ce", [(70000, 96, 6), (4099, 96, 3), (513, 128, 8)])
def test_adj_head_output_layer(M, E, ce):
    g = torch.Generator(device=DEV).manual_seed(M)
    h = torch.randn(M, E, device=DEV, generator=g).to(torch.bfloat16)
    w = torch.randn(ce, E, device=DEV, generator=g) / E ** 0.5
    b = torch.randn(ce, device=DEV, generator=g)
    dtok = torch.randn(M, ce, device=DEV, generator=g)
    tok = torch.empty(M, ce, device=DEV)
    dw = torch.full((ce, E), 0.25, device=DEV)
    lib, st = native.lib(), native.stream_ptr(DEV)
    native.check(lib.dsg_tr_adj_fc2(h.data_ptr(), w.data_ptr(), b.data_ptr(), tok.data_ptr(), None, None, M, E, ce, st), "fwd")
    native.check(lib.dsg_tr_adj_fc2(h.data_ptr(), None, None, None, dtok.data_ptr(), dw.data_ptr(), M, E, ce, st), "wgrad")
    assert _rel(tok, h.float() @ w.t() + b) < 1e-5
    assert _rel(dw - 0.25, dtok.t() @ h.float()) < 1e-4


# ---------------------------------------------------------------------------------------------------------
# window attention backward
# ---------------------------------------------------------------------------------------------------------
def _attention_reference(qkv, bias, mask, batch, res, w, shift, heads):
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


@pytest.mark.parametrize("batch,res,w,shift,heads", [(3, 16, 4, 0, 3), (3, 8, 4, 2, 6), (2, 64, 8, 0, 3), (5, 16, 8, 4, 12),
                                                      (2, 8, 8, 0, 24), (2, 20, 10, 5, 6), (3, 10, 10, 0, 12), (40, 16, 8, 0, 6)])
def test_window_attention_backward(batch, res, w, shift, heads):
    g = torch.Generator(device=DEV).manual_seed(res * 100 + w + shift)
    c, t = heads * 32, w * w
    qkv = torch.randn(batch * res * res, 3 * c, device=DEV, generator=g)
    qkv[:, :c] *= 32 ** -0.5
    qkv = qkv.to(torch.bfloat16)
    datt = torch.randn(batch * res * res, c, device=DEV, generator=g).to(torch.bfloat16)
    table = torch.randn((2 * w - 1) ** 2, heads, device=DEV, generator=g) * 0.5
    index = relative_position_index(w).to(DEV)
    mask = shifted_window_mask(res, w, shift).to(DEV) if shift else None
    q32 = qkv.float().requires_grad_(True)
    tab = table.clone().requires_grad_(True)
    bias_ref = tab[index.reshape(-1)].view(t, t, heads).permute(2, 0, 1)
    (_attention_reference(q32, bias_ref, mask, batch, res, w, shift, heads) * datt.float()).sum().backward()
    o = _ops()
    bias = torch.empty(heads, t, t, device=DEV)
    native.check(native.lib().dsg_tr_bias_gather(table.data_ptr(), index.data_ptr(), bias.data_ptr(), heads, t, 0, None, o.st),
                 "bias_gather")
    assert torch.equal(bias, bias_ref.detach().contiguous())
    dqkv = torch.empty_like(qkv)
    dbias = torch.zeros(heads, t, t, device=DEV)
    native.check(native.lib().dsg_tr_window_attention_bwd(qkv.data_ptr(), datt.data_ptr(), bias.data_ptr(), native.ptr(mask),
                                                          dqkv.data_ptr(), dbias.data_ptr(), batch, res, w, shift, heads,
                                                          o.st), "attention_bwd")
    dtable = torch.zeros_like(table)
    native.check(native.lib().dsg_tr_bias_gather(None, index.data_ptr(), dbias.data_ptr(), heads, t, 1, dtable.data_ptr(), o.st),
                 "bias_scatter")
    torch.cuda.synchronize()
    # bf16 operands of the tensor-core products (P and dS are rounded like the forward's P) and of the stored gradient
    assert _rel(dqkv.float(), q32.grad) < 1e-2, _rel(dqkv.float(), q32.grad)
    assert _rel(dtable, tab.grad) < 2e-3, _rel(dtable, tab.grad)     # fp32 dS from bf16-operand S / dP tiles


# ---------------------------------------------------------------------------------------------------------
# optimiser
# ---------------------------------------------------------------------------------------------------------
def test_fused_adam_ema_matches_torch():
    n = 100004                   # the flat buffers are multiples of 4 floats
    g = torch.Generator(device=DEV).manual_seed(3)
    p = torch.randn(n, device=DEV, generator=g)
    ref = p.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=2e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
    m, v = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    ema, ema_ref = p.clone(), p.clone()
    gs = torch.zeros(1, device=DEV)
    lib, st = native.lib(), native.stream_ptr(DEV)
    for step in range(1, 4):
        grad = torch.randn(n, device=DEV, generator=g) * (5.0 if step == 2 else 0.01)
        ref.grad = grad.clone()
        torch.nn.utils.clip_grad_norm_([ref], max_norm=10.0)
        opt.step()
        ema_ref.lerp_(ref.detach(), 1 - 0.9)
        native.check(lib.dsg_tr_sumsq(grad.data_ptr(), n, gs.data_ptr(), st), "sumsq")
        ptrs = (C.c_void_p * 8)(ema.data_ptr())
        dec = (C.c_float * 8)(0.9)
        native.check(lib.dsg_tr_adam_ema(p.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), n, gs.data_ptr(), 2e-3, 0.9,
                                         0.999, 1e-8, 0.01, step, 10.0, 1, ptrs, dec, st), "adam")
        assert _rel(gs.sqrt(), grad.norm()[None]) < 1e-5
        assert _rel(p, ref.detach()) < 1e-6 and _rel(ema, ema_ref) < 1e-6


# ---------------------------------------------------------------------------------------------------------
# the whole denoiser: parameter gradients against autograd of the CPU oracle
# ---------------------------------------------------------------------------------------------------------
def _net(cfg, sd):
    net = DiffuseSG(img_size=cfg["img"], in_chans=in_chans(cfg), patch_size=1, embed_dim=cfg["embed"], depths=cfg["depths"],
                    num_heads=[3, 6, 12, 24], window_size=cfg["window"], mlp_ratio=4., drop_rate=0., attn_drop_rate=0.,
                    drop_path_rate=0.0, self_condition=True, symmetric_noise=False, out_chans_adj=cfg["c_e"],
                    out_chans_node=cfg["c_n"])
    net.load_state_dict(sd, strict=True)
    return net.to(DEV)


def _oracle_grads(cfg, sd, adj, node, flags, sigmas, sc_adj, sc_node, wa, wn):
    """Gradients of sum(wa * D_adj) + sum(wn * D_node) w.r.t. every floating-point entry of the state dict, torch
    autograd through the fp32 CPU oracle of the preconditioned denoiser."""
    leaves = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "attn_mask" not in k else v) for k, v in sd.items()}

    def net(a, x, f, c_noise, sa, sn):
        return O.denoiser_forward(leaves, img=cfg["img"], embed=cfg["embed"], depths=cfg["depths"], heads=cfg["heads"],
                                  window=cfg["window"], self_condition=True, adj=a, node=x, flags=f, noise_labels=c_noise,
                                  sc_adj=sa, sc_node=sn)
    da, dn = O.precond_forward(net, adj, node, flags, sigmas, sc_adj, sc_node)
    ((da * wa).sum() + (dn * wn).sum()).backward()
    return da.detach(), dn.detach(), {k: v.grad for k, v in leaves.items() if v.is_floating_point() and v.requires_grad}


@pytest.mark.parametrize("name,batch", [("tiny", 4), ("vg", 2), ("coco", 4)])
def test_denoiser_parameter_gradients_match_oracle_autograd(name, batch):
    cfg = CONFIGS[name]
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    adj, node, flags, sigmas, sc_adj, sc_node = synthetic_inputs(cfg, batch, seed=11)
    sigmas = torch.tensor([0.2, 1.5, 4.0, 0.7])[:batch].contiguous()      # one noise level per sample, as in training
    g = torch.Generator().manual_seed(5)
    wa, wn = torch.randn(adj.shape, generator=g), torch.randn(node.shape, generator=g)
    ref_a, ref_n, ref_g = _oracle_grads(cfg, sd, adj, node, flags, sigmas, sc_adj, sc_node, wa, wn)
    net = _net(cfg, sd).train()
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=False, symmetric_noise=False).train()   # no coin flip here
    da, dn = model(adj.to(DEV), node.to(DEV), flags.to(DEV), sigmas.to(DEV), sc_adj.to(DEV), sc_node.to(DEV))
    assert da.requires_grad and dn.requires_grad
    ea, en = _rel(da.detach().cpu(), ref_a), _rel(dn.detach().cpu(), ref_n)
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
        d = (got.detach().cpu().double() - gr.double())
        num += float(d.pow(2).sum())
        den += float(gr.double().pow(2).sum())
        worst.append((float(d.norm() / gr.double().norm().clamp_min(1e-30)), k, float(gr.norm())))
    worst.sort(reverse=True)
    total = (num / den) ** 0.5
    print(f"{name}: outputs {ea:.2e} / {en:.2e}; all-parameter gradient rel-L2 {total:.3e}; worst " +
          ", ".join(f"{k} {e:.2e}" for e, k, _ in worst[:5]))
    # tolerance: bf16 GEMM operands in both directions.  The reference's OWN bf16-autocast gradients (torch CPU autocast of
    # the oracle, same inputs) sit 4.4e-2 (tiny) / 4.5e-2 (VG) from its fp32 gradients; measured here: 2.8e-2 / 3.1e-2
    assert total < 4e-2, (total, worst[:8])
    # every tensor whose gradient is not negligible next to the largest one agrees on its own as well
    gmax = max(n for _, _, n in worst)
    for e, k, n in worst:
        if n > 1e-3 * gmax:
            assert e < 1e-1, (k, e)


def test_training_step_runs_and_learns():
    """Twelve iterations of the reference's training step (objective -> model -> loss -> backward -> clip -> Adam -> EMAs) on
    one fixed batch: the loss falls, the moving averages follow ema_pytorch's schedule, eval() sees the new weights."""
    cfg = CONFIGS["tiny"]
    torch.manual_seed(0)
    np.random.seed(0)
    net = _net(cfg, synthetic_state_dict(cfg, seed=1234, stress=False)).train()
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).train()
    opt = FusedAdam(model, lr=1e-3, weight_decay=0.0, max_grad_norm=10.0)
    emas = [NativeEMA(model, beta=b) for b in (0.9, 0.99)]
    opt.attach_emas(emas)
    gen = NodeAdjEDMObjectiveGenerator("edm", "edm", dev=DEV, symmetric_noise=False)
    loss_fn = NodeAdjRainbowLoss(edge_loss_weight=1.0, node_loss_weight=1.0, objective="edm")
    B = 8
    adj, node, flags, *_ = synthetic_inputs(cfg, B, seed=3)
    adj, node = adj.sign(), node.clamp(-1, 1)
    adj = O.mask_pairs(adj, flags)
    node = O.mask_rows(node, flags)
    launches0 = native.launch_count()
    losses = []
    for it in range(12):
        torch.manual_seed(100)        # the same noise draw every iteration: a fixed regression problem
        la, ln = train_one_step(model, opt, emas, gen, loss_fn, adj, node, flags)
        losses.append(float(la.mean() + ln.mean()))
    assert native.launch_count() - launches0 > 1000
    assert all(np.isfinite(losses)) and losses[-1] < 0.97 * losses[0], losses
    # monotone up to the last-bit spread of the atomically accumulated gradients
    assert max(b - a for a, b in zip(losses, losses[1:])) < 1e-3 * losses[0], losses
    p = net.state_dict()["down_layers.0.blocks.0.mlp.fc1.weight"]
    e = emas[0].denoiser.state_dict()["down_layers.0.blocks.0.mlp.fc1.weight"]
    assert not torch.equal(p, e) and _rel(e, p) < 0.5
    # eval after training uses the updated weights (the inference arena is refreshed)
    model.eval()
    with torch.no_grad():
        np.random.seed(1)
        da, dn = model(adj.to(DEV), node.to(DEV), flags.to(DEV), torch.full((B,), 0.5, device=DEV))
    sd_now = {k: v.detach().cpu() for k, v in net.state_dict().items()}

    def onet(a, x, f, c, sa, sn):
        return O.denoiser_forward(sd_now, img=cfg["img"], embed=cfg["embed"], depths=cfg["depths"], heads=cfg["heads"],
                                  window=cfg["window"], self_condition=True, adj=a, node=x, flags=f, noise_labels=c,
                                  sc_adj=sa, sc_node=sn)
    np.random.seed(1)
    wa, wn = O.precond_forward(onet, adj, node, flags, torch.full((B,), 0.5), coin=np.random.rand)
    assert _rel(da.cpu(), wa) < 2.5e-2 and _rel(dn.cpu(), wn) < 2.5e-2


def test_fused_adam_step_matches_torch_adam_on_the_model():
    cfg = CONFIGS["tiny"]
    sd = synthetic_state_dict(cfg, seed=7, stress=True)
    net = _net(cfg, sd).train()
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=False, symmetric_noise=False).train()
    opt = FusedAdam(model, lr=1e-3, weight_decay=0.0, max_grad_norm=10.0)
    adj, node, flags, sigmas, sc_adj, sc_node = synthetic_inputs(cfg, 4, seed=2)
    opt.zero_grad(set_to_none=True)
    da, dn = model(adj.to(DEV), node.to(DEV), flags.to(DEV), sigmas.to(DEV))
    (da.square().mean() + dn.square().mean()).backward()
    before = {k: v.detach().clone() for k, v in net.named_parameters()}
    grads = {k: v.grad.detach().clone() for k, v in net.named_parameters()}
    ref = [before[k].clone().requires_grad_(True) for k in before]
    for r, k in zip(ref, before):
        r.grad = grads[k].clone()
    ropt = torch.optim.Adam(ref, lr=1e-3)
    torch.nn.utils.clip_grad_norm_(ref, max_norm=10.0)
    ropt.step()
    opt.step()
    for r, (k, v) in zip(ref, net.named_parameters()):
        assert _rel(v.detach(), r.detach()) < 1e-6, k


def test_training_kernels_ignore_shared_memory_leftovers():
    """Forward + backward of the training step with all shared memory overwritten by NaN patterns after every launch: the
    outputs are unchanged and the gradients stay within the run-to-run spread of their atomic accumulation order."""
    cfg = CONFIGS["tiny"]
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    adj, node, flags, sigmas, sc_adj, sc_node = [t.to(DEV) for t in synthetic_inputs(cfg, 4, seed=11)]
    sigmas = torch.tensor([0.2, 1.5, 4.0, 0.7], device=DEV)
    res = []
    for poison in (0, 1):
        net = _net(cfg, sd).train()
        model = NodeAdjPrecond(precond="edm", model=net, self_condition=False, symmetric_noise=False).train()
        native.lib().dsg_debug_set_smem_poison(0x7fc00000, poison)
        try:
            da, dn = model(adj, node, flags, sigmas, sc_adj, sc_node)
            (da.square().mean() + dn.square().mean()).backward()
            torch.cuda.synchronize()
        finally:
            native.lib().dsg_debug_set_smem_poison(0, 0)
        res.append((da.detach().clone(), dn.detach().clone(), train_state(net, DEV).grad.clone()))
    (a0, n0, g0), (a1, n1, g1) = res
    assert torch.equal(a0, a1) and torch.equal(n0, n1)
    assert torch.isfinite(g1).all() and _rel(g1, g0) < 1e-4, _rel(g1, g0)


def test_graphed_training_step_matches_eager():
    """One CUDA graph per iteration (objective + forward + loss + backward, both coin outcomes) against the eager launch
    sequence: same seeds per step, same coin stream -> the same losses and weights up to the order of the atomic gradient
    accumulations."""
    cfg = CONFIGS["tiny"]
    adj, node, flags, *_ = synthetic_inputs(cfg, 8, seed=3)
    adj, node = O.mask_pairs(adj.sign(), flags).to(DEV), O.mask_rows(node.clamp(-1, 1), flags).to(DEV)
    flags = flags.to(DEV)
    runs = []
    for graphed in (False, True):
        net = _net(cfg, synthetic_state_dict(cfg, seed=1234, stress=False)).train()
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
    assert np.allclose(l0, l1, rtol=2e-3), (l0, l1)       # measured 2e-4; Adam amplifies the atomics' last-bit spread
    # Adam turns the last-bit differences of the atomically accumulated gradients into lr-sized differences wherever a
    # gradient is ~ eps (two eager runs differ the same way): 8 steps x lr 1e-3 against weights of std 0.02
    assert _rel(w1, w0) < 5e-3 and _rel(e1, e0) < 5e-3, (_rel(w1, w0), _rel(e1, e0))


def test_training_trajectory_matches_the_reference_loop():
    """Six optimiser steps of the reference's training loop (objective -> preconditioned model with its no-grad
    self-conditioning pass -> rainbow loss -> backward -> clip 10 -> Adam) on the native path and on the fp32 CPU oracle with
    torch autograd + torch.optim.Adam, fed the SAME noise draws, sigmas and coins: the loss trajectories coincide and the
    accumulated weight updates point the same way."""
    cfg = CONFIGS["tiny"]
    sd = synthetic_state_dict(cfg, seed=99, stress=True)
    B, steps, lr = 4, 6, 1e-3
    adj, node, flags, *_ = synthetic_inputs(cfg, B, seed=3)
    adj, node = O.mask_pairs(adj.sign(), flags), O.mask_rows(node.clamp(-1, 1), flags)
    net = _net(cfg, sd).train()
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).train()
    opt = FusedAdam(model, lr=lr, max_grad_norm=10.0)
    gen = NodeAdjEDMObjectiveGenerator("edm", "edm", dev=DEV, symmetric_noise=False)
    loss_fn = NodeAdjRainbowLoss(edge_loss_weight=1.0, node_loss_weight=1.0, objective="edm")
    leaves = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "attn_mask" not in k else v) for k, v in sd.items()}
    ref_params = [v for v in leaves.values() if v.is_floating_point() and v.requires_grad]
    ref_opt = torch.optim.Adam(ref_params, lr=lr)

    def onet(a, x, f, c_noise, sa, sn):
        return O.denoiser_forward(leaves, img=cfg["img"], embed=cfg["embed"], depths=cfg["depths"], heads=cfg["heads"],
                                  window=cfg["window"], self_condition=True, adj=a, node=x, flags=f, noise_labels=c_noise,
                                  sc_adj=sa, sc_node=sn)
    rng = np.random.RandomState(7)
    coins = [bool(rng.rand() < 0.5) for _ in range(steps)]
    assert any(coins) and not all(coins)
    adj_d, node_d, flags_d = adj.to(DEV), node.to(DEV), flags.to(DEV)
    got, want = [], []
    for k in range(steps):
        torch.manual_seed(100 + k)
        na, nx, cond, ta, tx, (c_skip, c_out, c_in, c_noise, sigmas, weights) = gen.get_input_output(adj_d, node_d, flags_d)
        # native
        model.__dict__["_forced_coin"] = coins[k]
        opt.zero_grad(set_to_none=True)
        oa, ox = model(adjs=na, nodes=nx, node_flags=flags_d, sigmas=sigmas)
        la, ln = loss_fn(net_pred_a=oa, net_pred_x=ox, net_target_a=ta, net_target_x=tx, net_cond=cond, adjs_perturbed=na,
                         adjs_gt=adj_d, x_perturbed=nx, x_gt=node_d, node_flags=flags_d, loss_weight=weights, reduction="none")
        (la.mean() + ln.mean()).backward()
        opt.step()
        got.append(float(la.mean() + ln.mean()))
        # reference loop on the oracle (model/precond/precond.py:90-105, trainer_node_adj.py:109-175)
        na_c, nx_c, sig_c, w_c = na.cpu(), nx.cpu(), sigmas.cpu(), weights.cpu()
        sa = sn = None
        if coins[k]:
            with torch.no_grad():
                sa, sn = O.precond_forward(onet, na_c, nx_c, flags, sig_c, None, None)
        da, dn = O.precond_forward(onet, na_c, nx_c, flags, sig_c, sa, sn)
        ra, rn = T.regression_loss(da, dn, ta.cpu(), tx.cpu(), flags, w_c, 1.0, 1.0, "none")
        ref_opt.zero_grad(set_to_none=True)
        (ra.mean() + rn.mean()).backward()
        torch.nn.utils.clip_grad_norm_(ref_params, max_norm=10.0)
        ref_opt.step()
        want.append(float(ra.mean() + rn.mean()))
    model.__dict__["_forced_coin"] = None
    print("loss trajectory native", [f"{v:.5f}" for v in got], "reference", [f"{v:.5f}" for v in want])
    # the loss inherits the bf16 rounding of the forward (F to ~1e-2 per pass, weighted by (sigma^2 + 1/4) / (sigma/2)^2)
    assert np.allclose(got, want, rtol=1e-2), (got, want)
    num = den_a = den_b = 0.0
    for key, p in net.named_parameters():
        da_ = (p.detach().cpu() - sd[key]).double().flatten()
        db_ = (leaves[key].detach() - sd[key]).double().flatten()
        num += float(da_ @ db_)
        den_a += float(da_ @ da_)
        den_b += float(db_ @ db_)
    cos = num / (den_a * den_b) ** 0.5
    print(f"cosine between the accumulated weight updates: {cos:.4f}")
    assert cos > 0.9, cos


@pytest.mark.parametrize("name,batch", [("tiny", 4), ("vg", 2)])
def test_training_gradients_match_reference_goldens(name, batch, golden_dir):
    """The native forward + backward of one training iteration (model -> rainbow loss -> backward) against gradients the
    UNMODIFIED reference produced on the same weights and inputs (tests/golden/make_golden_train.py): losses, the norm of
    every parameter's gradient, and the complete gradient of the tensors the fixture holds."""
    import os
    cfg = CONFIGS[name]
    g = np.load(os.path.join(golden_dir, f"train_grads_{name}.npz"))
    sd = synthetic_state_dict(cfg, seed=1234, stress=True)
    adj, node, flags, _, sc_adj, sc_node = synthetic_inputs(cfg, batch, seed=11)
    sigmas = torch.tensor([0.2, 1.5, 4.0, 0.7, 0.05, 9.0, 0.9, 2.2])[:batch].contiguous()
    f = flags.float()
    tgt_adj = adj.sign() * f[:, None, :, None] * f[:, None, None, :]
    tgt_node = node.clamp(-1, 1) * f[:, :, None]
    weights = (sigmas ** 2 + 0.25) / (sigmas * 0.5) ** 2
    net = _net(cfg, sd).train()
    model = NodeAdjPrecond(precond="edm", model=net, self_condition=False, symmetric_noise=False).train()
    loss_fn = NodeAdjRainbowLoss(edge_loss_weight=1.0, node_loss_weight=1.0, objective="edm")
    dev = lambda t: t.to(DEV)
    oa, ox = model(adjs=dev(adj), nodes=dev(node), node_flags=dev(flags), sigmas=dev(sigmas), self_cond_adjs=dev(sc_adj),
                   self_cond_nodes=dev(sc_node))
    la, ln = loss_fn(net_pred_a=oa, net_pred_x=ox, net_target_a=dev(tgt_adj), net_target_x=dev(tgt_node), net_cond=dev(sigmas),
                     adjs_perturbed=dev(adj), adjs_gt=dev(tgt_adj), x_perturbed=dev(node), x_gt=dev(tgt_node),
                     node_flags=dev(flags), loss_weight=dev(weights), reduction="none")
    (la.mean() + ln.mean()).backward()
    torch.cuda.synchronize()
    assert np.allclose(la.detach().cpu().numpy(), g["loss_adj"], rtol=3e-2) and np.allclose(ln.detach().cpu().numpy(), g["loss_node"], rtol=3e-2)
    params = dict(net.named_parameters())
    norms = g["norms"]
    big = norms.max()
    worst = 0.0
    for k, want in zip(list(g["keys"]), norms):
        got = float(params[k].grad.double().norm())
        if want > 1e-3 * big:
            worst = max(worst, abs(got - want) / want)
            assert abs(got - want) < 6e-2 * want, (k, got, want)
    errs = {}
    for key in g.files:
        if key.startswith("grad::"):
            want = torch.from_numpy(g[key])
            errs[key[6:]] = _rel(params[key[6:]].grad.detach().cpu(), want)
    print(f"{name}: worst gradient-norm deviation {worst:.2e}; full tensors: " + ", ".join(f"{k} {e:.2e}" for k, e in errs.items()))
    assert max(errs.values()) < 1e-1 and float(np.mean(list(errs.values()))) < 4e-2, errs
