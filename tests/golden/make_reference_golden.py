"""Golden vectors produced by the REFERENCE'S OWN CODE for the pieces of the path that can run here.

The reference (``/root/reference``) cannot be imported as a package: ``nets/__init__`` pulls in e3nn's tensor-product
machinery, torch_scatter, torch_cluster and torch_geometric, none of which exists in this image.  Five of its modules
need nothing of e3nn beyond ``o3.Irreps`` (parsing), the ``compile_mode`` decorator and ``normalize2mom``:

    nets/gaussian_rbf.py    GaussianRadialBasisLayer                 (pure torch)
    nets/expnorm_rbf.py     ExpNormalSmearing, CosineCutoff          (pure torch)
    nets/radial_func.py     RadialProfile                            (pure torch once imported)
    nets/layer_norm.py      EquivariantLayerNormV2                   (Irreps + compile_mode)
    nets/fast_activation.py Activation                               (Irreps + compile_mode + normalize2mom)

This script imports exactly those files from where they lie, behind a stub ``e3nn`` whose ``o3.Irreps`` is this
repository's ``Irreps`` (used for nothing but "how many copies of which degree, in which order"), runs them in float64
on seeded inputs and writes inputs, ``state_dict`` and outputs to ``tests/golden/reference_modules.npz``.  The
arithmetic in the fixture is therefore the reference's, statement for statement; ``normalize2mom`` inside
``Activation`` is the one exception (our restatement of e3nn's Monte-Carlo constant) and the fixture says so.

A second fixture, ``reference_model_small.npz``, runs the reference's WHOLE model file
(``nets/graph_attention_transformer.py``: embeddings, ``TransBlock`` / ``GraphAttention`` / ``FeedForwardNetwork``, the
tensor-product wrappers of ``tensor_product_rescale.py``, gates, drop paths, readout) on a two-molecule batch with small
channel counts.  There the third-party calls the file makes - ``o3.TensorProduct``, ``o3.spherical_harmonics``,
``o3.ElementwiseTensorProduct``, ``e3nn.nn.Gate``, ``torch_scatter.scatter``, ``torch_geometric.utils.softmax``,
``torch_cluster.radius_graph`` - are served by stubs built on the ORACLE's restatements of those libraries
(``oracle/e3nn_ref.py``), so this fixture pins the oracle's restatement of the reference's own files (instruction lists,
irreps sorting, rescale / bias handling, head reshapes, attention wiring, residuals, scale factors), not the third-party
numerics underneath, which stay "parity unpinned".  With the same stubs the script also writes
  * ``reference_model_md17_small.npz``  - the MD17 model file (Lmax = 3, exp-normal basis, forces by autograd),
  * ``reference_model_headline.npz``    - the headline configuration at full size (3.53 M parameters; large tensors are a
                                          closed form of (name, shape, mean, std), see tests/helpers.closed_form_tensor),
  * ``reference_block_oc20_l1.npz``     - one TransBlock at the OC20 IS2RE l1_256_nonlinear sizes,
  * ``reference_state_shapes.json``     - parameter / buffer names and shapes of every registered configuration that does
                                          not need ocpmodels' Bessel basis, from the reference's constructors,
and, inside ``reference_modules.npz``, training-mode outputs of the dropout / stochastic-depth modules of ``drop.py``.

Run in the build container only (``python tests/golden/make_reference_golden.py``); the GPU box has no
``/root/reference`` and only ever reads the committed ``.npz`` files.  No reference source is copied anywhere.
"""
from __future__ import annotations

import importlib
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference/nets"


def _stub_e3nn():
    sys.path.insert(0, ROOT)
    from equiformer_b200 import o3 as our_o3
    from equiformer_b200.math import normalize2mom

    e3nn = types.ModuleType("e3nn")
    o3 = types.ModuleType("e3nn.o3")
    o3.Irreps = our_o3.Irreps
    o3.Irrep = our_o3.Irrep
    util = types.ModuleType("e3nn.util")
    jit = types.ModuleType("e3nn.util.jit")
    jit.compile_mode = lambda _mode: (lambda cls: cls)
    argtools = types.ModuleType("e3nn.util._argtools")        # Activation probes the parity of its functions on this device
    argtools._get_device = lambda _mod: torch.device("cpu")
    emath = types.ModuleType("e3nn.math")
    emath.normalize2mom = normalize2mom
    e3nn.__path__, util.__path__ = [], []
    e3nn.o3, e3nn.util, e3nn.math, util.jit, util._argtools = o3, util, emath, jit, argtools
    for name, mod in (("e3nn", e3nn), ("e3nn.o3", o3), ("e3nn.util", util), ("e3nn.util.jit", jit),
                      ("e3nn.util._argtools", argtools), ("e3nn.math", emath)):
        sys.modules[name] = mod


def _triples(irreps):
    """our Irreps (or a string) -> the oracle's [(mul, l, p)]"""
    from equiformer_b200 import o3 as our_o3
    return [(mul, ir.l, ir.p) for mul, ir in our_o3.Irreps(irreps)]


def _stub_third_party():
    """Everything nets/graph_attention_transformer.py imports besides torch, served by the oracle's restatements."""
    from collections import namedtuple

    from equiformer_b200 import o3 as our_o3
    from oracle import e3nn_ref as e3
    from oracle import equiformer_ref as R

    e3nn, o3 = sys.modules["e3nn"], sys.modules["e3nn.o3"]
    Instruction = namedtuple("Instruction", "i_in1 i_in2 i_out connection_mode has_weight path_weight path_shape")

    class TensorProduct(torch.nn.Module):       # the slice of e3nn 0.4.4's o3.TensorProduct the reference touches
        def __init__(self, irreps_in1, irreps_in2, irreps_out, instructions, normalization=None, internal_weights=None,
                     shared_weights=None, path_normalization="element"):
            super().__init__()
            assert path_normalization == "none" and normalization in (None, "component")
            self.irreps_in1, self.irreps_in2, self.irreps_out = (our_o3.Irreps(i) for i in (irreps_in1, irreps_in2, irreps_out))
            ins = []
            for t in instructions:
                i1, i2, io, mode, has_w = t[:5]
                m1, m2, mo = self.irreps_in1[i1].mul, self.irreps_in2[i2].mul, self.irreps_out[io].mul
                shape = {"uvw": (m1, m2, mo), "uvu": (m1, m2)}[mode]
                ins.append(Instruction(i1, i2, io, mode, has_w, float(self.irreps_out[io].ir.dim) ** 0.5, shape))
            self.instructions = ins
            self.weight_numel = sum(int(np.prod(i.path_shape)) for i in ins if i.has_weight)
            if shared_weights is False and internal_weights is None:
                internal_weights = False
            if shared_weights is None:
                shared_weights = True
            if internal_weights is None:
                internal_weights = shared_weights and self.weight_numel > 0
            self.internal_weights, self.shared_weights = internal_weights, shared_weights
            if internal_weights and self.weight_numel > 0:
                self.weight = torch.nn.Parameter(torch.randn(self.weight_numel))
            else:
                self.register_buffer("weight", torch.Tensor())

        def weight_views(self):
            off = 0
            for i in self.instructions:
                n = int(np.prod(i.path_shape))
                yield self.weight[off:off + n].view(i.path_shape)
                off += n

        def forward(self, x, y, weight=None):
            w = self.weight if weight is None else weight
            assert all(i.has_weight for i in self.instructions)
            # NodeEmbeddingNetwork hands over `one_hot(...).float()` (:686): exact in any dtype, evaluated in the weights'
            x, y = x.to(w.dtype), y.to(w.dtype)
            return e3.tensor_product(x, y, w, _triples(self.irreps_in1), _triples(self.irreps_in2), _triples(self.irreps_out),
                                     [(i.i_in1, i.i_in2, i.i_out, i.connection_mode) for i in self.instructions],
                                     self.shared_weights)

    class ElementwiseTensorProduct(torch.nn.Module):     # irreps x scalars, multiplicity by multiplicity
        def __init__(self, irreps_in1, irreps_in2):
            super().__init__()
            self.irreps_in1, self.irreps_in2 = our_o3.Irreps(irreps_in1).simplify(), our_o3.Irreps(irreps_in2).simplify()
            assert all(ir.l == 0 for _, ir in self.irreps_in2) and self.irreps_in1.num_irreps == self.irreps_in2.num_irreps
            self.irreps_out = self.irreps_in1

        def forward(self, x, y):
            out, off, g = [], 0, 0
            for mul, ir in self.irreps_in1:
                blk = x[..., off:off + mul * ir.dim].reshape(*x.shape[:-1], mul, ir.dim)
                out.append((blk * y[..., g:g + mul].unsqueeze(-1)).reshape(*x.shape[:-1], mul * ir.dim))
                off, g = off + mul * ir.dim, g + mul
            return torch.cat(out, dim=-1)

    def spherical_harmonics(l, x, normalize, normalization="integral"):
        ls = [l] if isinstance(l, int) else [ir.l for _, ir in our_o3.Irreps(l)]
        return e3.spherical_harmonics(ls, x, normalize, normalization)

    o3.TensorProduct, o3.ElementwiseTensorProduct, o3.spherical_harmonics = TensorProduct, ElementwiseTensorProduct, spherical_harmonics

    class Gate(torch.nn.Module):                 # e3nn.nn.Gate: SiLU on the scalars, sigmoid gates on the rest
        def __init__(self, irreps_scalars, act_scalars, irreps_gates, act_gates, irreps_gated):
            super().__init__()
            self.s, self.g, self.v = (our_o3.Irreps(i) for i in (irreps_scalars, irreps_gates, irreps_gated))
            assert act_scalars == [torch.nn.functional.silu] and (len(self.g) == 0 or act_gates == [torch.sigmoid])
            self.irreps_in = (self.s + self.g + self.v)
            self.irreps_out = self.s + self.v

        def forward(self, x):
            return R.gate(x, _triples(self.s), _triples(self.g), _triples(self.v))

    class NNActivation(torch.nn.Module):         # e3nn.nn.Activation on scalars only (all the reference asks of it)
        def __init__(self, irreps_in, acts):
            super().__init__()
            self.irreps_in = self.irreps_out = our_o3.Irreps(irreps_in)
            assert acts == [torch.nn.functional.silu] and all(ir.l == 0 for _, ir in self.irreps_in)

        def forward(self, x):
            return torch.nn.functional.silu(x) * e3.NORMALIZE2MOM["silu"]

    nn = types.ModuleType("e3nn.nn")
    nn.Gate, nn.Activation = Gate, NNActivation
    e3nn.nn = nn
    gp = types.ModuleType("e3nn.nn.models.v2106.gate_points_message_passing")

    def tp_path_exists(irreps_in1, irreps_in2, ir_out):
        ir_out = our_o3.Irrep(ir_out)
        return any(ir_out in ir1 * ir2 for _, ir1 in our_o3.Irreps(irreps_in1).simplify() for _, ir2 in our_o3.Irreps(irreps_in2).simplify())

    gp.tp_path_exists = tp_path_exists
    perm = types.ModuleType("e3nn.math.perm")
    perm.inverse = lambda p: tuple(int(i) for i in np.argsort(np.asarray(p)))
    sys.modules["e3nn.math"].perm = perm
    chain = {"e3nn.nn": nn, "e3nn.nn.models": types.ModuleType("e3nn.nn.models"),
             "e3nn.nn.models.v2106": types.ModuleType("e3nn.nn.models.v2106"),
             "e3nn.nn.models.v2106.gate_points_message_passing": gp, "e3nn.math.perm": perm}
    for name, mod in chain.items():
        mod.__path__ = []
        sys.modules[name] = mod

    tc = types.ModuleType("torch_cluster")
    tc.radius_graph = lambda pos, r, batch, max_num_neighbors=32: torch.stack(R.radius_graph(pos, r, batch))
    ts = types.ModuleType("torch_scatter")

    def scatter(src, index, dim=0, out=None, dim_size=None, reduce="sum"):
        assert dim == 0 and out is None and reduce == "sum"
        return R.scatter_sum(src, index, int(index.max()) + 1 if dim_size is None else dim_size)

    ts.scatter = scatter
    tg, tgnn, tgu, tgi = (types.ModuleType(n) for n in ("torch_geometric", "torch_geometric.nn", "torch_geometric.utils",
                                                        "torch_geometric.nn.inits"))

    def glorot(t):
        bound = (6.0 / (t.size(-2) + t.size(-1))) ** 0.5
        with torch.no_grad():
            t.uniform_(-bound, bound)

    tgi.glorot = glorot
    tgu.softmax = lambda src, index, ptr=None, num_nodes=None: R.pyg_softmax(src, index, int(index.max()) + 1 if num_nodes is None else num_nodes)
    tgu.degree = lambda index, num_nodes=None, dtype=None: torch.zeros(num_nodes, dtype=dtype).index_add_(0, index, torch.ones(index.shape[0], dtype=dtype))
    tgnn.global_mean_pool = tgnn.global_max_pool = None
    tgnn.inits, tg.nn, tg.utils = tgi, tgnn, tgu
    oc = {n: types.ModuleType(n) for n in ("ocpmodels", "ocpmodels.models", "ocpmodels.models.gemnet", "ocpmodels.models.gemnet.layers",
                                           "ocpmodels.models.gemnet.layers.radial_basis")}
    oc["ocpmodels.models.gemnet.layers.radial_basis"].RadialBasis = type("RadialBasis", (torch.nn.Module,), {})
    for name, mod in {"torch_cluster": tc, "torch_scatter": ts, "torch_geometric": tg, "torch_geometric.nn": tgnn,
                      "torch_geometric.utils": tgu, "torch_geometric.nn.inits": tgi, **oc}.items():
        mod.__path__ = []
        sys.modules[name] = mod


def _reference_module(name: str):
    """Import /root/reference/nets/<name>.py as ``refnets.<name>`` without executing nets/__init__.py."""
    if "refnets" not in sys.modules:
        pkg = types.ModuleType("refnets")
        pkg.__path__ = [REF]
        sys.modules["refnets"] = pkg
    return importlib.import_module(f"refnets.{name}")


def _randomise(module: torch.nn.Module, gen: torch.Generator, scale: float = 0.5):
    """Move every parameter off its initial value so that weights, biases and offsets all matter.  The module is still
    float32 here: parameters (and inputs) are float32 numbers evaluated in float64, so the fixture stores them in 4 bytes."""
    with torch.no_grad():
        for p in module.parameters():
            p.add_(scale * torch.randn(p.shape, generator=gen, dtype=p.dtype))
    return module.double()


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t.float().double()


def _store(dst: dict, prefix: str, module: torch.nn.Module, **arrays):
    for k, v in module.state_dict().items():
        assert torch.equal(v.float().double(), v.double()), k
        dst[f"{prefix}/state/{k}"] = v.detach().float().cpu().numpy()
    for k, v in arrays.items():
        if isinstance(v, torch.Tensor):
            exact32 = k != "y" and torch.equal(v.float().double(), v)
            dst[f"{prefix}/{k}"] = (v.float() if exact32 else v).detach().cpu().numpy()
        else:
            dst[f"{prefix}/{k}"] = np.asarray(v)


def main():
    if not os.path.isdir(REF):
        raise SystemExit(f"{REF} is not here: this generator runs in the build container only")
    _stub_e3nn()
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(1234)
    out: dict = {}

    # ---- Gaussian radial basis (gaussian_rbf.py:12-40), the configuration of every shipped model: 128 functions, 5 A
    # mean / std keep the reference's own initialisation (uniform, std >= 1/128 - perturbing std towards zero makes
    # (x - mean) / std a float32-hostile quotient in ANY implementation); the scalar weight and bias are moved off 1 and 0
    m = _reference_module("gaussian_rbf").GaussianRadialBasisLayer(128, 5.0)
    with torch.no_grad():
        m.weight.fill_(1.0625)
        m.bias.fill_(-0.03125)
    m = m.double()
    # the per-row cases store only their leading rows (the full draw keeps the stream of the later cases), so the
    # fixture stays under 1 MB
    dist = _f32(0.2 + 4.8 * torch.rand(67, generator=gen, dtype=torch.float64))[:32]
    _store(out, "gaussian_rbf", m, dist=dist, y=m(dist), num_basis=128, cutoff=5.0)

    # ---- exp-normal smearing + cosine cutoff (expnorm_rbf.py:5-78), the MD17 default basis
    m = _reference_module("expnorm_rbf").ExpNormalSmearing(0.0, 5.0, 32, False).double()
    dist = _f32(0.1 + 5.2 * torch.rand(99, generator=gen, dtype=torch.float64))      # some beyond the cutoff
    _store(out, "expnorm_rbf", m, dist=dist, y=m(dist), num_rbf=32, cutoff=5.0)

    # ---- radial profile (radial_func.py:9-51): Linear -> LayerNorm -> SiLU, twice, Linear without bias, + offset
    for tag, ch in (("qm9", [128, 64, 64, 960]), ("small", [32, 64, 64, 96])):
        m = _randomise(_reference_module("radial_func").RadialProfile(ch), gen, 0.2)
        x = _f32(torch.randn(19, ch[0], generator=gen, dtype=torch.float64))[:8 if tag == "qm9" else 19]
        _store(out, f"radial_profile_{tag}", m, x=x, y=m(x), ch_list=ch)

    # ---- equivariant layer norm (layer_norm.py:62-152) on the three node layouts of the shipped configurations
    LN = _reference_module("layer_norm").EquivariantLayerNormV2
    for tag, irreps in (("qm9_l2", "128x0e+64x1e+32x2e"), ("md17_l3", "128x0e+64x1o+64x2e+32x3o"), ("oc20_l1", "256x0e+128x1e"),
                        ("ffn_mid", "384x0e+192x1e+96x2e")):
        m = _randomise(LN(irreps), gen, 0.3)
        x = _f32(torch.randn(13, m.irreps.dim, generator=gen, dtype=torch.float64))[:6]
        _store(out, f"layer_norm_{tag}", m, x=x, y=m(x), eps=m.eps)
        out[f"layer_norm_{tag}/irreps"] = np.asarray(irreps)

    # ---- scalar activation (fast_activation.py:15-87); normalize2mom here is OUR restatement (see module docstring)
    Act = _reference_module("fast_activation").Activation
    m = Act("48x0e+16x0o", [torch.nn.SiLU(), torch.tanh])
    x = _f32(torch.randn(23, 64, generator=gen, dtype=torch.float64))
    out["activation/x"] = x.float().numpy()
    out["activation/y"] = m(x).detach().numpy()
    out["activation/irreps"] = np.asarray("48x0e+16x0o")

    # ---- stochastic depth and equivariant dropout (drop.py:31-106) in TRAINING mode: same torch seed, same draws.
    # EquivariantDropout multiplies through o3.ElementwiseTensorProduct, which here is the plain per-multiplicity product
    # (the only thing that product can be for scalar masks in 'component' normalisation)
    _stub_third_party()
    drop = _reference_module("drop")
    node_irreps = sys.modules["e3nn.o3"].Irreps("128x0e+64x1e+32x2e")
    x = _f32(torch.randn(31, 480, generator=torch.Generator().manual_seed(99), dtype=torch.float64)).float()   # own stream, the cases below keep their draws
    batch31 = torch.repeat_interleave(torch.arange(5), torch.tensor([7, 6, 6, 5, 7]))
    out["drop/x"], out["drop/batch"] = x.numpy(), batch31.numpy()
    for tag, module, args in (("drop_path", drop.DropPath(0.3), (x,)), ("graph_drop_path", drop.GraphDropPath(0.4), (x, batch31)),
                              ("equivariant_dropout", drop.EquivariantDropout(node_irreps, 0.25), (x,)),
                              ("scalars_dropout", drop.EquivariantScalarsDropout(node_irreps, 0.25), (x,))):
        module.train()
        torch.manual_seed(321)
        out[f"drop/{tag}"] = module(*args).numpy()

    path = os.path.join(HERE, "reference_modules.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path) / 1024:.0f} KiB")

    # ---- the reference's model file end to end, small channel counts, third-party calls served by the oracle
    _stub_third_party()
    gat = _reference_module("graph_attention_transformer")
    cfg = dict(irreps_in="5x0e", irreps_node_embedding="16x0e+8x1e+4x2e", num_layers=2, irreps_node_attr="1x0e",
               irreps_sh="1x0e+1x1e+1x2e", max_radius=5.0, number_of_basis=16, fc_neurons=[16, 16], irreps_feature="32x0e",
               irreps_head="8x0e+4x1e+2x2e", num_heads=2, irreps_pre_attn=None, rescale_degree=False, nonlinear_message=True,
               irreps_mlp_mid="24x0e+12x1e+6x2e", norm_layer="layer", alpha_drop=0.0, proj_drop=0.0, out_drop=0.0,
               drop_path_rate=0.0)
    torch.manual_seed(7)
    model = gat.GraphAttentionTransformer(**cfg)
    with torch.no_grad():                      # biases, offsets and norm shifts start at zero: move them
        for name, prm in model.named_parameters():
            if prm.abs().max() == 0 or "bias" in name or "offset" in name:
                prm.add_(0.1 * torch.randn(prm.shape, generator=gen))
    torch.set_default_dtype(torch.float64)     # the forward creates one-hot / ones tensors in the default dtype
    model = model.double().eval()
    n_atoms = [7, 5]
    batch = torch.repeat_interleave(torch.arange(2), torch.tensor(n_atoms))
    pos = _f32(2.2 * torch.randn(sum(n_atoms), 3, generator=gen, dtype=torch.float64))
    z = torch.tensor([6, 1, 1, 8, 7, 1, 9, 6, 6, 8, 1, 1])
    taps = {}
    hooks = [model.edge_deg_embed.register_forward_hook(lambda m, i, o: taps.__setitem__("edge_deg_embed", o.detach())),
             model.blocks[0].ga.register_forward_hook(lambda m, i, o: taps.__setitem__("blocks.0.ga", o.detach())),
             model.blocks[0].register_forward_hook(lambda m, i, o: taps.__setitem__("blocks.0", o.detach()))]
    with torch.no_grad():
        energy = model(f_in=None, pos=pos, batch=batch, node_atom=z)
    for h in hooks:
        h.remove()
    model.zero_grad()
    (model(f_in=None, pos=pos, batch=batch, node_atom=z) ** 2).sum().backward()        # d(sum E^2) / d(parameters)
    grads = {f"grad/{k}": p.grad.detach().numpy() for k, p in model.named_parameters() if p.grad is not None}
    small = {f"state/{k}": v.detach().float().numpy() if v.is_floating_point() else v.numpy()
             for k, v in model.state_dict().items() if v is not None}
    small.update(grads)
    for k, v in model.state_dict().items():
        if v is not None and v.is_floating_point():
            assert torch.equal(v.float().double(), v), k
    small.update({"pos": pos.float().numpy(), "batch": batch.numpy(), "z": z.numpy(), "energy": energy.numpy(),
                  **{f"tap/{k}": v.numpy() for k, v in taps.items()}})
    for k, v in cfg.items():
        if v is not None:
            small[f"cfg/{k}"] = np.asarray(v)
    path = os.path.join(HERE, "reference_model_small.npz")
    np.savez_compressed(path, **small)
    print(f"wrote {path}: {len(small)} arrays, {os.path.getsize(path) / 1024:.0f} KiB; energy {energy.flatten().tolist()}")

    # ---- the MD17 model file (energy + forces by autograd, Lmax = 3, exp-normal basis), same stubs
    torch.set_default_dtype(torch.float32)
    md = _reference_module("graph_attention_transformer_md17")
    cfg = dict(irreps_in="64x0e", irreps_node_embedding="16x0e+8x1e+4x2e+4x3e", num_layers=2, irreps_node_attr="1x0e",
               irreps_sh="1x0e+1x1e+1x2e+1x3e", max_radius=5.0, number_of_basis=16, basis_type="exp", fc_neurons=[16, 16],
               irreps_feature="32x0e", irreps_head="8x0e+4x1e+2x2e+2x3e", num_heads=2, irreps_pre_attn=None,
               rescale_degree=False, nonlinear_message=True, irreps_mlp_mid="24x0e+12x1e+6x2e+6x3e", norm_layer="layer",
               alpha_drop=0.0, proj_drop=0.0, out_drop=0.0, drop_path_rate=0.0)
    torch.manual_seed(11)
    model = md.GraphAttentionTransformerMD17(**cfg)
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if prm.abs().max() == 0 or "bias" in name or "offset" in name:
                prm.add_(0.1 * torch.randn(prm.shape, generator=gen))
    torch.set_default_dtype(torch.float64)
    model = model.double().eval()
    z = torch.tensor([6, 6, 8, 1, 1, 1, 1, 6, 8])
    batch = torch.zeros(9, dtype=torch.long)
    pos = _f32(1.8 * torch.randn(9, 3, generator=gen, dtype=torch.float64))
    energy, forces = model(node_atom=z, pos=pos.clone(), batch=batch)
    model.zero_grad()
    (energy.sum() + (forces ** 2).sum()).backward()            # energy + force loss: a second derivative through the forward
    grads = {f"grad/{k}": p.grad.detach().numpy() for k, p in model.named_parameters() if p.grad is not None}
    small = {f"state/{k}": v.detach().float().numpy() if v.is_floating_point() else v.numpy()
             for k, v in model.state_dict().items() if v is not None}
    small.update(grads)
    for k, v in model.state_dict().items():
        if v is not None and v.is_floating_point():
            assert torch.equal(v.float().double(), v), k
    small.update({"pos": pos.float().numpy(), "batch": batch.numpy(), "z": z.numpy(), "energy": energy.detach().numpy(),
                  "forces": forces.detach().numpy()})
    for k, v in cfg.items():
        if v is not None:
            small[f"cfg/{k}"] = np.asarray(v)
    path = os.path.join(HERE, "reference_model_md17_small.npz")
    np.savez_compressed(path, **small)
    print(f"wrote {path}: {len(small)} arrays, {os.path.getsize(path) / 1024:.0f} KiB; energy {energy.flatten().tolist()}")
    torch.set_default_dtype(torch.float32)

    # ---- the HEADLINE configuration at its real size (3.53 M parameters).  Large tensors are replaced by a closed form of
    # (name, shape, mean, std) that the tests rebuild (tests/helpers.closed_form_tensor), small ones are stored verbatim
    from tests.helpers import closed_form_tensor
    torch.manual_seed(3)
    model = gat.graph_attention_transformer_nonlinear_l2(irreps_in="5x0e", radius=5.0, num_basis=128)
    head = {}
    with torch.no_grad():
        for k, v in model.state_dict().items():
            if v is None or not v.is_floating_point() or v.numel() == 0:
                continue
            if v.numel() <= 1024:
                if v.abs().max() == 0:
                    v.add_(0.05 * torch.randn(v.shape, generator=gen))
                head[f"small/{k}"] = v.detach().float().numpy().copy()
            else:
                mean, std = float(v.mean()), float(v.std())
                head[f"stat/{k}"] = np.asarray([mean, std], dtype=np.float64)
                v.copy_(closed_form_tensor(k, v.shape, mean, std))
    torch.set_default_dtype(torch.float64)
    model = model.double().eval()
    n_atoms = [9, 7]
    batch = torch.repeat_interleave(torch.arange(2), torch.tensor(n_atoms))
    pos = _f32(1.9 * torch.randn(sum(n_atoms), 3, generator=gen, dtype=torch.float64))
    z = torch.tensor([6, 1, 1, 8, 7, 1, 9, 6, 1, 6, 6, 8, 1, 1, 7, 1])
    taps = {}
    hook = model.blocks[0].register_forward_hook(lambda m, i, o: taps.__setitem__("blocks.0", o.detach()))
    with torch.no_grad():
        energy = model(f_in=None, pos=pos, batch=batch, node_atom=z)
    hook.remove()
    torch.set_default_dtype(torch.float32)
    head.update({"pos": pos.float().numpy(), "batch": batch.numpy(), "z": z.numpy(), "energy": energy.numpy(),
                 "tap/blocks.0": taps["blocks.0"].numpy()})
    path = os.path.join(HERE, "reference_model_headline.npz")
    np.savez_compressed(path, **head)
    print(f"wrote {path}: {len(head)} arrays, {os.path.getsize(path) / 1024:.0f} KiB; energy {energy.flatten().tolist()}")

    # ---- the dot-product-attention variant (nets/dp_attention_transformer.py), small configuration, energy + parameter
    # gradients: the q.k logits replace the MLP attention, everything else is the same machinery
    dp = _reference_module("dp_attention_transformer")
    cfg = dict(irreps_in="5x0e", irreps_node_embedding="16x0e+8x1e+4x2e", num_layers=2, irreps_node_attr="1x0e",
               irreps_sh="1x0e+1x1e+1x2e", max_radius=5.0, number_of_basis=16, fc_neurons=[16, 16], irreps_feature="32x0e",
               irreps_head="8x0e+4x1e+2x2e", num_heads=2, irreps_pre_attn=None, rescale_degree=False, nonlinear_message=False,
               irreps_mlp_mid="24x0e+12x1e+6x2e", norm_layer="layer", alpha_drop=0.0, proj_drop=0.0, out_drop=0.0,
               drop_path_rate=0.0)
    torch.manual_seed(13)
    model = dp.DotProductAttentionTransformer(**cfg)
    g3 = torch.Generator().manual_seed(4321)
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if prm.abs().max() == 0 or "bias" in name or "offset" in name:
                prm.add_(0.1 * torch.randn(prm.shape, generator=g3))
    torch.set_default_dtype(torch.float64)
    model = model.double().eval()
    n_atoms = [6, 7]
    batch = torch.repeat_interleave(torch.arange(2), torch.tensor(n_atoms))
    pos = _f32(2.0 * torch.randn(sum(n_atoms), 3, generator=g3, dtype=torch.float64))
    z = torch.tensor([6, 1, 8, 1, 7, 1, 6, 6, 9, 1, 1, 8, 1])
    energy = model(f_in=None, pos=pos, batch=batch, node_atom=z)
    model.zero_grad()
    (energy ** 2).sum().backward()
    torch.set_default_dtype(torch.float32)
    small = {f"state/{k}": v.detach().float().numpy() if v.is_floating_point() else v.numpy()
             for k, v in model.state_dict().items() if v is not None}
    for k, v in model.state_dict().items():
        if v is not None and v.is_floating_point():
            assert torch.equal(v.float().double(), v), k
    small.update({f"grad/{k}": p.grad.detach().numpy() for k, p in model.named_parameters() if p.grad is not None})
    small.update({"pos": pos.float().numpy(), "batch": batch.numpy(), "z": z.numpy(), "energy": energy.detach().numpy()})
    for k, v in cfg.items():
        if v is not None:
            small[f"cfg/{k}"] = np.asarray(v)
    path = os.path.join(HERE, "reference_model_dp_small.npz")
    np.savez_compressed(path, **small)
    print(f"wrote {path}: {len(small)} arrays, {os.path.getsize(path) / 1024:.0f} KiB; energy {energy.flatten().tolist()}")

    # ---- the dot-product variant of the MD17 model (nets/dp_attention_transformer_md17.py): energy, forces, gradients
    dpm = _reference_module("dp_attention_transformer_md17")
    cfg = dict(irreps_in="64x0e", irreps_node_embedding="16x0e+8x1e+4x2e+4x3e", num_layers=2, irreps_node_attr="1x0e",
               irreps_sh="1x0e+1x1e+1x2e+1x3e", max_radius=5.0, number_of_basis=16, basis_type="exp", fc_neurons=[16, 16],
               irreps_feature="32x0e", irreps_head="8x0e+4x1e+2x2e+2x3e", num_heads=2, irreps_pre_attn=None,
               rescale_degree=False, nonlinear_message=False, irreps_mlp_mid="24x0e+12x1e+6x2e+6x3e", norm_layer="layer",
               alpha_drop=0.0, proj_drop=0.0, out_drop=0.0, drop_path_rate=0.0)
    torch.manual_seed(17)
    model = dpm.DotProductAttentionTransformerMD17(**cfg)
    g4 = torch.Generator().manual_seed(8765)
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if prm.abs().max() == 0 or "bias" in name or "offset" in name:
                prm.add_(0.1 * torch.randn(prm.shape, generator=g4))
    torch.set_default_dtype(torch.float64)
    model = model.double().eval()
    z = torch.tensor([6, 8, 1, 1, 6, 1, 8, 1])
    batch = torch.zeros(8, dtype=torch.long)
    pos = _f32(1.7 * torch.randn(8, 3, generator=g4, dtype=torch.float64))
    energy, forces = model(node_atom=z, pos=pos.clone(), batch=batch)
    model.zero_grad()
    (energy.sum() + (forces ** 2).sum()).backward()
    torch.set_default_dtype(torch.float32)
    small = {f"state/{k}": v.detach().float().numpy() if v.is_floating_point() else v.numpy()
             for k, v in model.state_dict().items() if v is not None}
    for k, v in model.state_dict().items():
        if v is not None and v.is_floating_point():
            assert torch.equal(v.float().double(), v), k
    small.update({f"grad/{k}": p.grad.detach().numpy() for k, p in model.named_parameters() if p.grad is not None})
    small.update({"pos": pos.float().numpy(), "batch": batch.numpy(), "z": z.numpy(), "energy": energy.detach().numpy(),
                  "forces": forces.detach().numpy()})
    for k, v in cfg.items():
        if v is not None:
            small[f"cfg/{k}"] = np.asarray(v)
    path = os.path.join(HERE, "reference_model_dp_md17_small.npz")
    np.savez_compressed(path, **small)
    print(f"wrote {path}: {len(small)} arrays, {os.path.getsize(path) / 1024:.0f} KiB; energy {energy.flatten().tolist()}")

    # ---- one transformer block at the OC20 IS2RE `l1_256_nonlinear` sizes (oc20/configs/is2re/all/graph_attention_transformer/
    # l1_256_nonlinear_g@2_local.yml: 256x0e+128x1e, 8 heads of 32x0e+16x1e, mlp 768x0e+384x1e, Lmax = 1).  The OC20 model
    # file itself needs ocpmodels; its blocks are the TransBlock class of graph_attention_transformer.py, run here.
    torch.manual_seed(5)
    kw = dict(irreps_node_input="256x0e+128x1e", irreps_node_attr="1x0e", irreps_edge_attr="1x0e+1x1e",
              irreps_node_output="256x0e+128x1e", fc_neurons=[128, 64, 64], irreps_head="32x0e+16x1e", num_heads=8,
              irreps_pre_attn="256x0e+128x1e", rescale_degree=False, nonlinear_message=True, alpha_drop=0.0, proj_drop=0.0,
              drop_path_rate=0.0, irreps_mlp_mid="768x0e+384x1e", norm_layer="layer")
    blk = gat.TransBlock(**kw)
    oc = {}
    with torch.no_grad():
        for k, v in blk.state_dict().items():
            if v is None or not v.is_floating_point() or v.numel() == 0:
                continue
            if v.numel() <= 1024:
                if v.abs().max() == 0:
                    v.add_(0.05 * torch.randn(v.shape, generator=gen))
                oc[f"small/{k}"] = v.detach().float().numpy().copy()
            else:
                mean, std = float(v.mean()), float(v.std())
                oc[f"stat/{k}"] = np.asarray([mean, std], dtype=np.float64)
                v.copy_(closed_form_tensor(k, v.shape, mean, std))
    oc["shapes"] = np.asarray(json.dumps({k: list(v.shape) for k, v in blk.state_dict().items() if v is not None}))
    torch.set_default_dtype(torch.float64)
    blk = blk.double().eval()
    n_nodes = 14
    g2 = torch.Generator().manual_seed(77)
    pos = 2.0 * torch.randn(n_nodes, 3, generator=g2, dtype=torch.float64)
    batch = torch.zeros(n_nodes, dtype=torch.long)
    edge_src, edge_dst = sys.modules["torch_cluster"].radius_graph(pos, 5.0, batch)
    edge_sh = sys.modules["e3nn.o3"].spherical_harmonics("1x0e+1x1e", pos[edge_src] - pos[edge_dst], True, "component")
    edge_scalars = _f32(torch.rand(edge_src.shape[0], 128, generator=g2, dtype=torch.float64))
    x = _f32(torch.randn(n_nodes, 640, generator=g2, dtype=torch.float64))
    edge_sh = _f32(edge_sh)
    with torch.no_grad():
        y = blk(node_input=x, node_attr=torch.ones(n_nodes, 1), edge_src=edge_src, edge_dst=edge_dst, edge_attr=edge_sh,
                edge_scalars=edge_scalars, batch=batch)
    torch.set_default_dtype(torch.float32)
    oc.update({"x": x.float().numpy(), "edge_src": edge_src.numpy(), "edge_dst": edge_dst.numpy(), "edge_sh": edge_sh.float().numpy(),
               "edge_scalars": edge_scalars.float().numpy(), "y": y.numpy()})
    for k, v in kw.items():
        if v is not None:
            oc[f"cfg/{k}"] = np.asarray(v)
    path = os.path.join(HERE, "reference_block_oc20_l1.npz")
    np.savez_compressed(path, **oc)
    print(f"wrote {path}: {len(oc)} arrays, {os.path.getsize(path) / 1024:.0f} KiB; E = {edge_src.shape[0]}, max|y| = {float(y.abs().max()):.3f}")

    # ---- every registered configuration that does not need ocpmodels' Bessel basis, at its real size: parameter and
    # buffer names with shapes, as the reference's constructors create them (no forward; a few KB of JSON)
    table = {}
    for mod, irreps_in, names in (
            (gat, "5x0e", ["graph_attention_transformer_l2", "graph_attention_transformer_nonlinear_l2",
                           "graph_attention_transformer_nonlinear_l2_e3"]),
            (md, "64x0e", ["graph_attention_transformer_l2_md17", "graph_attention_transformer_nonlinear_l2_md17",
                           "graph_attention_transformer_nonlinear_l2_e3_md17", "graph_attention_transformer_nonlinear_exp_l2_md17",
                           "graph_attention_transformer_nonlinear_exp_l3_md17", "graph_attention_transformer_nonlinear_attn_exp_l3_md17",
                           "graph_attention_transformer_nonlinear_exp_l3_e3_md17"]),
            (dp, "5x0e", ["dot_product_attention_transformer_l2"]),
            (dpm, "64x0e", ["dot_product_attention_transformer_exp_l2_md17", "dot_product_attention_transformer_exp_l3_md17"])):
        for name in names:
            model = getattr(mod, name)(irreps_in=irreps_in, radius=5.0, num_basis=128)
            table[name] = {k: list(v.shape) for k, v in model.state_dict().items() if v is not None}
            print(f"  {name}: {len(table[name])} entries, {sum(p.numel() for p in model.parameters())} parameters")
    path = os.path.join(HERE, "reference_state_shapes.json")
    with open(path, "w") as f:
        json.dump(table, f, indent=0, sort_keys=True)
    print(f"wrote {path}: {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
