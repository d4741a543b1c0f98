"""Full-length golden vectors from the UNMODIFIED reference (build container only; ~25 min of CPU).

    python tests/golden/make_golden_full.py [precond] [sampler] [decode]

What it runs (everything imported from /root/reference where it lies, nothing copied):

* ``precond``  - ``NodeAdjPrecond.forward`` (model/precond/precond.py:65-110) on the Visual Genome and COCO-Stuff
  geometries, four noise levels, the coin-flip stream included  ->  precond_{vg,coco}.npz
* ``sampler``  - ``NodeAdjEDMSampler.sample`` (runner/mcmc_sampler/edm.py:291-445), **256 steps, batch 8**, on the
  CPU device, so that the initial noise, the 2 x 256 per-step ``randn_like`` draws and the numpy coin flips all come
  from the two global generators seeded below.  A test replays the identical streams with
  ``torch.manual_seed`` / ``np.random.seed`` and a ``torch.randn_like`` that draws on the CPU generator, so no noise
  is committed - only the reference's OUTPUTS: the final state of all 8 graphs and 10 interim snapshots (every 32
  steps) of the first two, stored without repeats (``save_sampler256``)  ->  sampler256_{vg,vg_refinit,coco}.npz
* ``decode``   - the reference's post-sampling decode.  ``_decode_node`` / ``_decode_adj`` are closures inside
  ``sg_go_sampling`` (runner/sampler/sampler_node_adj.py:222-285) whose module cannot be imported here
  (evaluation.* needs pyemd); their source text is lifted out of the file with ``ast`` and compiled against the
  reference's own ``mask_adjs`` / ``mask_nodes`` (utils/graph_utils.py) and ``bin2dec`` (utils/attribute_code.py:319),
  i.e. the reference's statements run unmodified.  Inputs: the final samples above plus a seeded edge-case tensor
  (exact zeros, values beyond +-1, bit patterns beyond the class range)  ->  decode_{vg,coco}.npz
"""
import ast
import os
import sys
import time
import zipfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from make_golden import REF, build_ref, import_reference  # noqa: E402

SAMPLER_CASES = {  # name -> (config, stress weights, batch, torch seed, numpy seed)
    "vg": ("vg", True, 8, 101, 101),
    "vg_refinit": ("vg", False, 8, 102, 102),
    "coco": ("coco", True, 8, 103, 103),
}
RAW_TYPES = {"vg": (150, 51), "coco": (171, 7)}   # (raw_num_node_type, raw_num_adj_type), utils/sg_utils.py:355-394


def make_precond(DiffuseSG, NodeAdjPrecond):
    from diffusesg_b200.utils.synthetic import CONFIGS, synthetic_inputs, synthetic_state_dict
    for name in ("vg", "coco"):
        cfg = CONFIGS[name]
        net = build_ref(DiffuseSG, cfg).eval()
        net.load_state_dict(synthetic_state_dict(cfg, seed=1234, stress=True), strict=True)
        model = NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).eval()
        adj, node, flags, _, _, _ = synthetic_inputs(cfg, 2, seed=7)
        np.random.seed(5)
        coins = np.random.rand(4)
        np.random.seed(5)
        out = {"coins": coins}
        sa = sn = None
        with torch.no_grad():
            for k, s in enumerate((40.0, 3.0, 0.4, 0.01)):
                sa, sn = model(adj * s, node * s, flags, torch.full((2,), s), sa, sn)
                out[f"adj_{k}"], out[f"node_{k}"] = sa.numpy().copy(), sn.numpy().copy()
        np.savez_compressed(os.path.join(HERE, f"precond_{name}.npz"), **out)
        print("precond", name, coins)


def save_sampler256(path, out):
    """Write a sampler256 golden under 1 MB without losing a compared value: of the ten adjacency snapshots only
    the eight after steps 0 - 224 are stored (``adjs_ls_mid``); the one after step 255 equals ``adjs[:2]`` and the
    initial noise is pinned through ``nodes_ls[0]`` (tests/conftest.py: sampler256_golden rebuilds ``adjs_ls``).
    The archive is an ordinary .npz, LZMA- instead of deflate-compressed; ``np.load`` reads it as is."""
    out = dict(out)
    adjs_ls = out.pop("adjs_ls")
    assert np.array_equal(adjs_ls[-1], out["adjs"][:2])
    out["adjs_ls_mid"] = adjs_ls[1:-1]
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as z:
        for key, val in out.items():
            with z.open(key + ".npy", "w") as f:
                np.lib.format.write_array(f, np.asanyarray(val), allow_pickle=False)


def make_sampler(DiffuseSG, NodeAdjPrecond, NodeAdjEDMSampler, only=None):
    from diffusesg_b200.utils.synthetic import CONFIGS, synthetic_node_flags, synthetic_state_dict
    for case, (name, stress, batch, tseed, nseed) in SAMPLER_CASES.items():
        if only and case not in only:
            continue
        cfg = CONFIGS[name]
        net = build_ref(DiffuseSG, cfg).eval()
        net.load_state_dict(synthetic_state_dict(cfg, seed=1234, stress=stress), strict=True)
        model = NodeAdjPrecond(precond="edm", model=net, self_condition=True, symmetric_noise=False).eval()
        flags = synthetic_node_flags(cfg, batch, seed=77)
        sampler = NodeAdjEDMSampler(num_steps=256, clip_samples=True, clip_samples_min=-1.0, clip_samples_max=1.0,
                                    clip_samples_scope="x_0", dev="cpu", objective="edm", self_condition=True,
                                    symmetric_noise=False)
        passes = [0]
        hook = net.register_forward_hook(lambda *_: passes.__setitem__(0, passes[0] + 1))
        torch.manual_seed(tseed)
        np.random.seed(nseed)
        t0 = time.time()
        a, n, a_ls, n_ls = sampler.sample(model=model, node_flags=flags, flag_interim_adjs=True,
                                          max_num_interim_adjs=9, num_node_chan=cfg["c_n"], num_edge_chan=cfg["c_e"])
        hook.remove()
        out = dict(adjs=a.numpy(), nodes=n.numpy(), adjs_ls=a_ls[:, :2].numpy(), nodes_ls=n_ls[:, :2].numpy(),
                   flags=flags.numpy(), raw_passes=np.int64(passes[0]), torch_seed=np.int64(tseed),
                   numpy_seed=np.int64(nseed), batch=np.int64(batch),
                   snapshot_steps=np.linspace(0, 256, 9).astype(int).clip(max=255))
        save_sampler256(os.path.join(HERE, f"sampler256_{case}.npz"), out)
        print("sampler256", case, "passes", passes[0], "%.0f s" % (time.time() - t0), a_ls.shape, n_ls.shape,
              "rms", float(a.pow(2).mean().sqrt()), flush=True)


def reference_decoders(raw_num_node_type, raw_num_adj_type):
    """The two closures of sg_go_sampling, compiled from the reference's own source text."""
    sys.path.insert(0, REF)
    from utils.attribute_code import attribute_converter, bin2dec
    from utils.graph_utils import mask_adjs, mask_nodes
    sys.path.remove(REF)
    path = os.path.join(REF, "runner/sampler/sampler_node_adj.py")
    tree = ast.parse(open(path).read())
    fns = [node for node in ast.walk(tree) if isinstance(node, ast.FunctionDef)
           and node.name in ("_decode_node", "_decode_adj")]
    assert sorted(f.name for f in fns) == ["_decode_adj", "_decode_node"]
    ns = dict(torch=torch, np=np, mask_adjs=mask_adjs, mask_nodes=mask_nodes, bin2dec=bin2dec,
              attribute_converter=attribute_converter, raw_num_node_type=raw_num_node_type,
              raw_num_adj_type=raw_num_adj_type, flag_node_only=False, flag_binary_edge=False)
    exec(compile(ast.Module(body=fns, type_ignores=[]), path, "exec"), ns)
    return ns["_decode_node"], ns["_decode_adj"], mask_nodes


def make_decode():
    from diffusesg_b200.utils.synthetic import CONFIGS, synthetic_node_flags
    for name in ("vg", "coco"):
        cfg = CONFIGS[name]
        n_types, a_types = RAW_TYPES[name]
        dec_node, dec_adj, mask_nodes = reference_decoders(n_types, a_types)
        out = {}
        cases = {}
        path = os.path.join(HERE, f"sampler256_{name}.npz")
        if os.path.exists(path):
            g = np.load(path)
            cases["final"] = (torch.from_numpy(g["adjs"]), torch.from_numpy(g["nodes"]), torch.from_numpy(g["flags"]))
        # seeded edge cases: zeros (sign threshold: > 0), beyond the clamp, every bit pattern incl. out-of-range ones
        gen = torch.Generator().manual_seed(9)
        flags = synthetic_node_flags(cfg, 6, seed=5)
        adj = torch.randn(6, cfg["c_e"], cfg["img"], cfg["img"], generator=gen) * 1.5
        node = torch.randn(6, cfg["img"], cfg["c_n"], generator=gen) * 1.5
        adj[0, :, :4] = 0.0
        adj[1] = adj[1].sign() * 3.0
        adj[2] = 1.0                       # all bits set: above the class range -> clamp
        node[0, :3] = 0.0
        node[2, :, :-4] = 1.0
        node[3] = node[3] * 4.0
        cases["edge"] = (adj, node, flags)
        for key, (a, n, f) in cases.items():
            q_node = dec_node(n[..., :-4].clone(), f, "bits")
            q_adj = dec_adj(a.clone(), f, "bits")
            bbox = mask_nodes((n[..., -4:] * 0.5 + 0.5).clone(), f)   # sampler_node_adj.py:202-209
            out[f"{key}_q_adj"], out[f"{key}_q_node"], out[f"{key}_bbox"] = q_adj.numpy(), q_node.numpy(), bbox.numpy()
            if key == "edge":
                out["edge_adj"], out["edge_node"], out["edge_flags"] = a.numpy(), n.numpy(), f.numpy()
            print("decode", name, key, q_adj.shape, q_node.shape, "max class", float(q_adj.max()), float(q_node.max()))
        np.savez_compressed(os.path.join(HERE, f"decode_{name}.npz"), **out)


if __name__ == "__main__":
    torch.set_num_threads(8)
    what = set(sys.argv[1:]) or {"precond", "sampler", "decode"}
    DiffuseSG, NodeAdjPrecond, NodeAdjEDMSampler = import_reference()
    if "precond" in what:
        make_precond(DiffuseSG, NodeAdjPrecond)
    if "sampler" in what:
        make_sampler(DiffuseSG, NodeAdjPrecond, NodeAdjEDMSampler,
                     only=[c for c in SAMPLER_CASES if c in what] or None)
    if "decode" in what:
        make_decode()
