"""Generate golden vectors by running the REFERENCE's own code (run in the build
container only; /root/reference does not exist on the GPU box).

    python tests/golden/make_golden.py            # writes tests/golden/*.pt

What is real and what is stubbed
--------------------------------
Loaded verbatim from /root/reference (never copied into this repo):
  hydragnn/utils/model/operations.py, hydragnn/models/Base.py,
  hydragnn/models/EGCLStack.py, hydragnn/models/PAINNStack.py, plus (AST-extracted,
  because their modules import absent packages at top level)
  ``activation_function_selection`` / ``loss_function_selection`` /
  ``unsorted_segment_mean`` from hydragnn/utils/model/model.py,
  ``EnhancedModelWrapper.energy_force_loss`` from hydragnn/models/create.py and
  ``RadiusGraphPBC._limit_neighbors`` / ``_remove_true_self_loops`` from
  hydragnn/preprocess/graph_samples_checks_and_updates.py.
Stubbed third-party packages that are absent from this image (semantics restated,
[3P-memory] in SURVEY.md Appendix B):
  torch_geometric.nn.Sequential (argument-string glue only), BatchNorm,
  global_{mean,add,max}_pool (index_add / amax), torch_scatter.scatter_add,
  hydragnn.utils.distributed.get_device (cpu), the tracer (no-op), GPSConv (unused).
So the E_GCL / PainnMessage / PainnUpdate / Base.forward / MLIP-loss arithmetic in the
golden files is the reference's own; only the glue named above is ours.
"""
import ast
import importlib.util
import os
import sys
import types

import numpy as np
import torch

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    if "." not in name or True:
        m.__path__ = []
    sys.modules[name] = m
    return m


def _extract(path, names, glb):
    """exec selected top-level (or nested) function/class definitions of a reference file."""
    tree = ast.parse(open(path).read())
    found = {}
    for node in ast.walk(tree):
        if isinstance(node, (ast.FunctionDef, ast.ClassDef)) and node.name in names and node.name not in found:
            found[node.name] = node
    for n in names:
        code = compile(ast.Module(body=[found[n]], type_ignores=[]), path, "exec")
        exec(code, glb)
    return glb


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


class StubSequential(torch.nn.Module):
    """[3P-memory B.5] torch_geometric.nn.Sequential: children are named module_<i>."""

    def __init__(self, input_args, modules):
        super().__init__()
        self.in_names = [a.strip() for a in input_args.split(",") if a.strip()]
        self.steps = []
        for i, item in enumerate(modules):
            fn, desc = item
            lhs, rhs = desc.split("->")
            if isinstance(fn, torch.nn.Module):
                self.add_module("module_%d" % i, fn)
            self.steps.append((fn, [a.strip() for a in lhs.split(",") if a.strip()],
                               [a.strip() for a in rhs.split(",") if a.strip()]))

    def forward(self, *args, **kwargs):
        env = dict(zip(self.in_names, args))
        env.update(kwargs)
        out = None
        for fn, ins, outs in self.steps:
            out = fn(*[env[k] for k in ins])
            if len(outs) == 1:
                env[outs[0]] = out
            else:
                for k, v in zip(outs, out):
                    env[k] = v
        return out


def _pool(kind):
    def f(x, batch, size=None):
        G = int(batch.max()) + 1 if size is None else size
        if kind == "add":
            return x.new_zeros(G, x.shape[1]).index_add_(0, batch, x)
        if kind == "mean":
            s = x.new_zeros(G, x.shape[1]).index_add_(0, batch, x)
            c = torch.bincount(batch, minlength=G).clamp(min=1).to(x.dtype)
            return s / c[:, None]
        out = x.new_full((G, x.shape[1]), float("-inf"))
        return out.scatter_reduce(0, batch[:, None].expand_as(x), x, reduce="amax")
    return f


def install_stubs():
    def scatter_add(src, index, dim=0):
        shape = list(src.shape)
        shape[dim] = int(index.max()) + 1
        return src.new_zeros(shape).index_add_(dim, index, src)

    _mod("torch_scatter", scatter_add=scatter_add, scatter=None)
    _mod("torch_geometric")
    _mod("torch_geometric.nn", Sequential=StubSequential, BatchNorm=torch.nn.BatchNorm1d,
         global_add_pool=_pool("add"), global_mean_pool=_pool("mean"), global_max_pool=_pool("max"))
    _mod("torch_geometric.typing", OptTensor=object)
    _mod("hydragnn")
    _mod("hydragnn.models")
    _mod("hydragnn.utils")
    _mod("hydragnn.utils.distributed", get_device=lambda *a, **k: torch.device("cpu"))
    _mod("hydragnn.utils.print")
    _mod("hydragnn.utils.print.print_utils", print_master=lambda *a, **k: None)
    _mod("hydragnn.utils.profiling_and_tracing")
    _mod("hydragnn.utils.profiling_and_tracing.tracer", start=lambda *a, **k: None, stop=lambda *a, **k: None)
    _mod("hydragnn.globalAtt")
    _mod("hydragnn.globalAtt.gps", GPSConv=None)
    glb = {"torch": torch}
    _extract(REF + "/hydragnn/utils/model/model.py",
             ["activation_function_selection", "loss_function_selection", "unsorted_segment_mean"], glb)
    _mod("hydragnn.utils.model", **{k: glb[k] for k in
                                    ("activation_function_selection", "loss_function_selection", "unsorted_segment_mean")})
    _load("hydragnn.utils.model.operations", REF + "/hydragnn/utils/model/operations.py")
    _load("hydragnn.models.Base", REF + "/hydragnn/models/Base.py")
    egcl = _load("hydragnn.models.EGCLStack", REF + "/hydragnn/models/EGCLStack.py")
    painn = _load("hydragnn.models.PAINNStack", REF + "/hydragnn/models/PAINNStack.py")
    return egcl, painn


def install_pnaeq_stubs():
    """PNAEqStack.py additionally needs PyG's MessagePassing / DegreeScalerAggregation / Linear / resolver.
    MessagePassing is used only as an nn.Module that stores ``aggr_module``; geom_Linear is nn.Linear with the
    same parameter names; DegreeScalerAggregation is the restatement in oracle/pnaeq.py (so the golden file pins
    everything in PNAEqStack.py EXCEPT that third-party aggregator)."""
    from oracle.pnaeq import DegreeScalerAggregation as OracleDSA

    class MessagePassing(torch.nn.Module):
        def __init__(self, aggr=None, node_dim=0, **kw):
            super().__init__()
            if aggr is not None:
                self.aggr_module = aggr

    class DSA(OracleDSA):
        def forward(self, x, index=None, dim_size=None, **kw):
            return super().forward(x, index, dim_size)

    tg = sys.modules["torch_geometric.nn"]
    tg.MessagePassing = MessagePassing
    tg.Linear = torch.nn.Linear
    _mod("torch_geometric.nn.resolver", activation_resolver=lambda act, **kw: {"tanh": torch.nn.Tanh}[act]())
    _mod("torch_geometric.nn.dense")
    _mod("torch_geometric.nn.dense.linear", Linear=torch.nn.Linear)
    _mod("torch_geometric.nn.aggr")
    _mod("torch_geometric.nn.aggr.scaler", DegreeScalerAggregation=DSA)
    sys.modules["torch_geometric.typing"].Adj = object
    sys.modules["torch_geometric"].nn = tg
    return _load("hydragnn.models.PNAEqStack", REF + "/hydragnn/models/PNAEqStack.py")


def install_gps_stubs():
    """gps.py needs PyG's PerformerAttention / MessagePassing / reset / resolvers / to_dense_batch.  Only
    ``to_dense_batch(x, None)`` (-> one sequence with an all-true mask, SURVEY B.3) and the ``batch_norm``
    normalisation (PyG BatchNorm = a module holding ``.module = BatchNorm1d``) are exercised."""
    from oracle.gps import PyGBatchNorm
    _mod("torch_geometric.nn.attention", PerformerAttention=type("PerformerAttention", (), {}))
    _mod("torch_geometric.nn.conv", MessagePassing=torch.nn.Module)
    _mod("torch_geometric.nn.inits", reset=lambda m: None)
    res = sys.modules.get("torch_geometric.nn.resolver") or _mod("torch_geometric.nn.resolver")
    res.activation_resolver = lambda act, **kw: {"tanh": torch.nn.Tanh, "relu": torch.nn.ReLU}[act]()
    res.normalization_resolver = lambda norm, channels, **kw: PyGBatchNorm(channels)
    sys.modules["torch_geometric.typing"].Adj = object
    _mod("torch_geometric.utils", to_dense_batch=lambda x, batch=None: (x.unsqueeze(0), torch.ones(1, x.shape[0], dtype=torch.bool)))
    gps = _load("hydragnn.globalAtt.gps", REF + "/hydragnn/globalAtt/gps.py")
    sys.modules["hydragnn.models.Base"].GPSConv = gps.GPSConv
    return gps


def install_mace_stubs():
    """The reference's MACE path = its own files (MACEStack.py, mace_utils/modules/{blocks,radial,symmetric_contraction}.py,
    mace_utils/tools/cg.py, irreps_tools.py) on top of e3nn 0.5.1, which is not installable here.  e3nn is replaced by the
    oracle's restatement (oracle/e3.py: Irreps, wigner_3j, SphericalHarmonics, Linear, TensorProduct "uvu", FullyConnectedNet);
    opt_einsum_fx (an einsum *optimiser*) by the identity; torch_scatter.scatter by index_add_; ase (only read by the distance
    transforms, unused here) by an empty module.  Everything else that runs is the reference's code."""
    from oracle import e3

    def scatter(src, index, dim=0, dim_size=None, reduce="sum"):
        n = int(index.max()) + 1 if dim_size is None else dim_size
        out = src.new_zeros((n,) + tuple(src.shape[1:])).index_add_(0, index, src)
        if reduce == "mean":
            cnt = torch.bincount(index, minlength=n).clamp(min=1).to(src.dtype)
            out = out / cnt.reshape((-1,) + (1,) * (src.dim() - 1))
        return out

    sys.modules["torch_scatter"].scatter = scatter
    o3 = _mod("e3nn.o3", Irreps=e3.Irreps, Irrep=e3.Irrep, Linear=e3.Linear, TensorProduct=e3.TensorProductUVU,
              SphericalHarmonics=e3.SphericalHarmonics, wigner_3j=e3.wigner_3j)
    nn_ = _mod("e3nn.nn", FullyConnectedNet=e3.FullyConnectedNet, Activation=type("Activation", (torch.nn.Module,), {}))
    _mod("e3nn", o3=o3, nn=nn_)
    _mod("e3nn.util")
    _mod("e3nn.util.jit", compile_mode=lambda mode: (lambda cls: cls))
    _mod("e3nn.util.codegen", CodeGenMixin=type("CodeGenMixin", (), {}))
    _mod("opt_einsum_fx", optimize_einsums_full=lambda model, example_inputs: model)
    ase = _mod("ase")
    ase.data = _mod("ase.data", covalent_radii=np.zeros(119))
    _mod("hydragnn.utils.model.mace_utils")
    _mod("hydragnn.utils.model.mace_utils.tools")
    _mod("hydragnn.utils.model.mace_utils.modules")
    _mod("hydragnn.utils.model.mace_utils.tools.compile", simplify_if_compile=lambda cls: cls)
    base = REF + "/hydragnn/utils/model"
    _load("hydragnn.utils.model.irreps_tools", base + "/irreps_tools.py")
    _load("hydragnn.utils.model.mace_utils.tools.cg", base + "/mace_utils/tools/cg.py")
    _load("hydragnn.utils.model.mace_utils.modules.radial", base + "/mace_utils/modules/radial.py")
    _load("hydragnn.utils.model.mace_utils.modules.symmetric_contraction", base + "/mace_utils/modules/symmetric_contraction.py")
    _load("hydragnn.utils.model.mace_utils.modules.blocks", base + "/mace_utils/modules/blocks.py")
    return _load("hydragnn.models.MACEStack", REF + "/hydragnn/models/MACEStack.py")


def toy_batch(gen, sizes, box, input_dim=1, dtype=torch.float32):
    """A few random molecules + an asymmetric hand-made edge list (every atom keeps its
    3 nearest in-graph neighbours as sources)."""
    from hydragnn_b200.data import Batch, Data
    samples = []
    for n in sizes:
        pos = torch.rand(n, 3, generator=gen, dtype=dtype) * box
        d = torch.cdist(pos, pos) + torch.eye(n, dtype=dtype) * 1e9
        k = min(3, n - 1)
        nbr = d.topk(k, largest=False).indices                        # [n, k]
        tgt = torch.arange(n)[:, None].expand(n, k)
        ei = torch.stack([nbr.reshape(-1), tgt.reshape(-1)]).long()
        x = torch.randint(1, 9, (n, input_dim), generator=gen).to(dtype)
        samples.append(Data(x=x, pos=pos, edge_index=ei,
                            edge_shifts=torch.zeros(ei.shape[1], 3, dtype=dtype),
                            energy=torch.randn(1, generator=gen, dtype=dtype),
                            forces=torch.randn(n, 3, generator=gen, dtype=dtype),
                            y=torch.randn(1, 1, generator=gen, dtype=dtype)))
    return Batch.from_data_list(samples)


def t2d(batch):
    return {k: v for k, v in batch.items() if torch.is_tensor(v)}


def main():
    egcl, painn = install_stubs()
    gen = torch.Generator().manual_seed(20260921)
    heads_node = {"node": [{"type": "branch-0", "architecture": {"num_headlayers": 2, "dim_headlayers": [12, 6], "type": "mlp"}}]}
    heads_graph = {"graph": [{"type": "branch-0", "architecture": {"num_sharedlayers": 2, "dim_sharedlayers": 5,
                                                                   "num_headlayers": 2, "dim_headlayers": [10, 7]}}]}

    # ---- layer level: E_GCL (plain + equivariant), PainnMessage, PainnUpdate ------------------
    out = {}
    b = toy_batch(gen, [5, 7, 4], 4.0, input_dim=6)
    for eq in (False, True):
        torch.manual_seed(1)
        layer = egcl.E_GCL(6, 10, 8, edge_attr_dim=0, equivariant=eq)
        res = layer(b.x, b.pos, b.edge_index, None, b.edge_shifts)
        out["egcl_eq%d" % eq] = {"state": layer.state_dict(), "x": b.x, "pos": b.pos, "edge_index": b.edge_index,
                                 "out": [r.detach() for r in (res if eq else (res,))]}
    torch.manual_seed(2)
    msg = painn.PainnMessage(node_size=6, num_radial=5, cutoff=7.0, edge_dim=None)
    upd = painn.PainnUpdate(node_size=6, last_layer=False)
    upd_last = painn.PainnUpdate(node_size=6, last_layer=True)
    ops = sys.modules["hydragnn.utils.model.operations"]
    diff, dist = ops.get_edge_vectors_and_lengths(b.pos, b.edge_index, b.edge_shifts, normalize=True)
    v0 = torch.randn(b.x.shape[0], 3, 6, generator=gen)
    s1, v1 = msg(b.x, v0, b.edge_index.t(), diff, dist)
    s2, v2 = upd(s1, v1)
    s3 = upd_last(s1, v1)
    out["painn_layer"] = {"msg_state": msg.state_dict(), "upd_state": upd.state_dict(), "upd_last_state": upd_last.state_dict(),
                          "x": b.x, "v": v0, "pos": b.pos, "edge_index": b.edge_index, "diff": diff, "dist": dist,
                          "sinc": painn.sinc_expansion(dist, 5, 7.0), "fcut": painn.cosine_cutoff(dist, 7.0),
                          "s1": s1.detach(), "v1": v1.detach(), "s2": s2.detach(), "v2": v2.detach(), "s3": s3.detach()}
    torch.save(out, HERE + "/layers.pt")

    # ---- full models through the reference's Base.forward -----------------------------------
    models = {}
    # (a) EGNN MLIP, node head, the C1/C3 shape in miniature
    b = toy_batch(gen, [6, 5, 8, 3], 4.0, input_dim=1)
    torch.manual_seed(0)
    m = egcl.EGCLStack("inv_node_feat, equiv_node_feat, edge_index, edge_attr, edge_shifts", "", None,
                       1, 16, [1], 0, "", "", 0, ["node"], heads_node, "relu", "mse", False,
                       max_neighbours=None, loss_weights=[1.0], freeze_conv=False, initial_bias=None,
                       num_conv_layers=3, num_nodes=None, graph_pooling="mean")
    m.eval()
    inp = t2d(b)
    b.pos.requires_grad_(True)
    pred = m(b)
    # the reference's own loss code, AST-extracted from the nested wrapper class
    glb = {"torch": torch, "torch_scatter": sys.modules["torch_scatter"]}
    _extract(REF + "/hydragnn/models/create.py", ["energy_force_loss"], glb)
    fake = types.SimpleNamespace(num_heads=1, head_type=["node"], model=m, loss_function=m.loss_function,
                                 energy_weight=1.0, energy_peratom_weight=1.0, force_weight=1.0)
    tot, tasks = glb["energy_force_loss"](fake, pred, b, create_graph=True)
    forces = -torch.autograd.grad(
        sys.modules["torch_scatter"].scatter_add(pred[0], b.batch, dim=0).sum(), b.pos, retain_graph=True)[0]
    grads = torch.autograd.grad(tot, list(m.parameters()), allow_unused=True)
    models["egnn_mlip"] = {"state": m.state_dict(), "inputs": inp, "pred": [p.detach() for p in pred],
                           "loss": tot.detach(), "tasks": [t.detach() for t in tasks], "forces": forces.detach(),
                           "grads": {n: (g.detach() if g is not None else None)
                                     for (n, _), g in zip(m.named_parameters(), grads)}}

    # (b) equivariant EGNN, graph + node heads
    b = toy_batch(gen, [6, 5, 8, 3], 4.0, input_dim=2)
    heads_both = dict(heads_graph, **heads_node)
    torch.manual_seed(0)
    m = egcl.EGCLStack("inv_node_feat, equiv_node_feat, edge_index, edge_attr, edge_shifts", "", None,
                       2, 12, [1, 3], 0, "", "", 0, ["graph", "node"], heads_both, "lrelu_01", "mse", True,
                       max_neighbours=None, loss_weights=[1.0, 2.0], freeze_conv=False, initial_bias=None,
                       num_conv_layers=3, num_nodes=None, graph_pooling="add")
    m.eval()
    pred = m(b)
    models["egnn_equiv_multihead"] = {"state": m.state_dict(), "inputs": t2d(b), "pred": [p.detach() for p in pred]}

    # (c) PaiNN, graph head, the C2 shape in miniature (input_dim = 1 -> first layer at width 1, quirk Q4)
    for pool in ("mean", "max"):
        b = toy_batch(gen, [9, 9, 7, 9], 5.0, input_dim=1)
        torch.manual_seed(0)
        m = painn.PAINNStack("inv_node_feat, equiv_node_feat, edge_index, diff, dist",
                             "inv_node_feat, equiv_node_feat, edge_index, diff, dist", None, 5, 7.0,
                             1, 16, [1], 0, "", "", 0, ["graph"], heads_graph, "relu", "mse", False,
                             loss_weights=[1.0], freeze_conv=False, num_conv_layers=2, num_nodes=None,
                             graph_pooling=pool)
        m.eval()
        pred = m(b)
        loss, _ = m.loss(pred, b.y, [torch.arange(b.y.shape[0])])
        grads = torch.autograd.grad(loss, list(m.parameters()), allow_unused=True)
        models["painn_graph_" + pool] = {"state": m.state_dict(), "inputs": t2d(b), "pred": [p.detach() for p in pred],
                                         "loss": loss.detach(),
                                         "grads": {n: (g.detach() if g is not None else None)
                                                   for (n, _), g in zip(m.named_parameters(), grads)}}
    torch.save(models, HERE + "/models.pt")

    # ---- PNAEq through the reference's PNAEqStack (third-party DegreeScalerAggregation restated, see stub) ----
    pna = install_pnaeq_stubs()
    pmodels = {}
    for pool, last_deg in (("mean", [0, 0, 0, 30, 0]), ("add", [0, 3, 0, 27, float("inf")])):
        b = toy_batch(gen, [9, 6, 7, 9], 5.0, input_dim=1)
        torch.manual_seed(0)
        m = pna.PNAEqStack("inv_node_feat, equiv_node_feat, edge_index, edge_rbf, edge_vec",
                           "inv_node_feat, equiv_node_feat, edge_index, edge_rbf, edge_vec", last_deg, None, 6, 5.0,
                           1, 12, [1], 0, "", "", 0, ["graph"], heads_graph, "relu", "mse", False,
                           loss_weights=[1.0], freeze_conv=False, num_conv_layers=3, num_nodes=None, graph_pooling=pool)
        m.eval()
        pred = m(b)
        loss, _ = m.loss(pred, b.y, [torch.arange(b.y.shape[0])])
        grads = torch.autograd.grad(loss, list(m.parameters()), allow_unused=True)
        pmodels["pnaeq_graph_" + pool] = {"state": m.state_dict(), "inputs": t2d(b), "pred": [p.detach() for p in pred],
                                          "loss": loss.detach(), "deg": last_deg,
                                          "grads": {n: (g.detach() if g is not None else None)
                                                    for (n, _), g in zip(m.named_parameters(), grads)}}
    torch.save(pmodels, HERE + "/models_pnaeq.pt")

    # ---- GPS: the reference's own gps.py + Base.py (PyG glue stubbed: BatchNorm wrapper, to_dense_batch, resolvers) ----
    gps = install_gps_stubs()
    gmodels = {}
    for kind in ("EGNN", "PAINN"):
        b = toy_batch(gen, [9, 6, 7, 9], 5.0, input_dim=2)
        b.pe = torch.randn(b.x.shape[0], 4, generator=gen)
        b.rel_pe = (b.pe[b.edge_index[0]] - b.pe[b.edge_index[1]]).abs()       # serialized_dataset_loader.py:186-189
        torch.manual_seed(0)
        if kind == "EGNN":
            m = egcl.EGCLStack("inv_node_feat, equiv_node_feat, edge_index, edge_attr, edge_shifts", "", None,
                               2, 16, [1], 4, "GPS", "multihead", 4, ["graph"], heads_graph, "relu", "mse", False,
                               max_neighbours=None, loss_weights=[1.0], freeze_conv=False, initial_bias=None,
                               num_conv_layers=2, num_nodes=None, graph_pooling="mean")
        else:
            m = painn.PAINNStack("inv_node_feat, equiv_node_feat, edge_index, diff, dist",
                                 "inv_node_feat, equiv_node_feat, edge_index, diff, dist", None, 5, 7.0,
                                 2, 16, [1], 4, "GPS", "multihead", 4, ["graph"], heads_graph, "relu", "mse", False,
                                 loss_weights=[1.0], freeze_conv=False, num_conv_layers=2, num_nodes=None, graph_pooling="mean")
        m.eval()
        pred_eval = [p.detach() for p in m(b)]
        # train mode (batch-statistics BatchNorm) with the dropout probabilities of THIS INSTANCE set to zero
        m.train()
        for mod in m.modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
            if isinstance(mod, gps.GPSConv):
                mod.dropout = 0.0
        state = {k: v.clone() for k, v in m.state_dict().items()}
        pred = m(b)
        loss, _ = m.loss(pred, b.y, [torch.arange(b.y.shape[0])])
        grads = torch.autograd.grad(loss, list(m.parameters()), allow_unused=True)
        gmodels["gps_" + kind.lower()] = {"state": state, "inputs": t2d(b), "pred_eval": pred_eval,
                                          "pred_train": [p.detach() for p in pred], "loss": loss.detach(),
                                          "state_after": {k: v.clone() for k, v in m.state_dict().items() if "running" in k},
                                          "grads": {n: (g.detach() if g is not None else None)
                                                    for (n, _), g in zip(m.named_parameters(), grads)}}
    torch.save(gmodels, HERE + "/models_gps.pt")

    # ---- RadiusGraphPBC numpy post-processing ---------------------------------------------
    glb = {"np": np}
    _extract(REF + "/hydragnn/preprocess/graph_samples_checks_and_updates.py",
             ["_limit_neighbors", "_remove_true_self_loops"], glb)
    rng = np.random.default_rng(7)
    E = 200
    src = rng.integers(0, 12, E)
    dst = rng.integers(0, 12, E)
    length = rng.random(E) * 5
    S = rng.integers(-1, 2, (E, 3))
    a = glb["_remove_true_self_loops"](None, src, dst, length, S)
    lim = glb["_limit_neighbors"](None, *a, 6)
    torch.save({"in": [torch.from_numpy(np.asarray(t)) for t in (src, dst, length, S)],
                "k": 6, "out": [torch.from_numpy(np.asarray(t)) for t in lim]}, HERE + "/pbc_limit.pt")
    # ---- node heads of type 'mlp_per_node' and 'conv' (Base.py:508-588, 648-680, 800-810, 912-979) -------------------
    # own generator so that the files above stay byte-identical; PyG BatchNorm naming (a module holding `.module`)
    from oracle.gps import PyGBatchNorm
    sys.modules["hydragnn.models.Base"].BatchNorm = PyGBatchNorm
    gen2 = torch.Generator().manual_seed(4321)
    hmodels, hmodels64 = {}, {}
    heads_pernode = {"node": [{"type": "branch-0", "architecture": {"num_headlayers": 2, "dim_headlayers": [7, 5], "type": "mlp_per_node"}}]}
    heads_conv = {"node": [{"type": "branch-0", "architecture": {"num_headlayers": 2, "dim_headlayers": [10, 6], "type": "conv"}}]}
    for name in ("egnn_mlp_per_node", "egnn_conv_head", "painn_conv_head"):
        b = toy_batch(gen2, [6, 6, 6] if name == "egnn_mlp_per_node" else [7, 5, 8], 4.0, input_dim=1)
        b.y = torch.randn(b.x.shape[0], 2, generator=gen2)
        torch.manual_seed(0)
        if name.startswith("egnn"):
            m = egcl.EGCLStack("inv_node_feat, equiv_node_feat, edge_index, edge_attr, edge_shifts", "", None,
                               1, 12, [2], 0, "", "", 0, ["node"], heads_pernode if name == "egnn_mlp_per_node" else heads_conv,
                               "relu", "mse", False, max_neighbours=None, loss_weights=[1.0], freeze_conv=False, initial_bias=None,
                               num_conv_layers=2, num_nodes=6 if name == "egnn_mlp_per_node" else None, graph_pooling="mean")
        else:
            m = painn.PAINNStack("inv_node_feat, equiv_node_feat, edge_index, diff, dist",
                                 "inv_node_feat, equiv_node_feat, edge_index, diff, dist", None, 5, 7.0,
                                 1, 12, [2], 0, "", "", 0, ["node"], heads_conv, "relu", "mse", False,
                                 loss_weights=[1.0], freeze_conv=False, num_conv_layers=2, num_nodes=None, graph_pooling="mean")
        m.train()                                      # batch-statistics BatchNorm in the conv heads
        state = {k: v.clone() for k, v in m.state_dict().items()}
        pred = m(b)
        loss, _ = m.loss(pred, b.y, [torch.arange(b.y.shape[0])])
        grads = torch.autograd.grad(loss, list(m.parameters()), allow_unused=True)
        hmodels[name] = {"state": state, "inputs": t2d(b), "pred": [p.detach() for p in pred], "loss": loss.detach(),
                         "grads": {n: (g.detach() if g is not None else None) for (n, _), g in zip(m.named_parameters(), grads)}}
        # the same weights and inputs in fp64: a conv head's batch-statistics BatchNorm over a few nodes amplifies fp32 rounding
        # to ~1e-5 relative, by an amount that depends on the host's BLAS kernels and thread count
        m.double()
        b64 = b.clone().to(dtype=torch.float64)
        pred = m(b64)
        loss, _ = m.loss(pred, b64.y, [torch.arange(b64.y.shape[0])])
        grads = torch.autograd.grad(loss, list(m.parameters()), allow_unused=True)
        hmodels64[name] = {"pred": [p.detach() for p in pred], "loss": loss.detach(),
                           "grads": {n: (g.detach() if g is not None else None) for (n, _), g in zip(m.named_parameters(), grads)}}
    torch.save(hmodels, HERE + "/models_heads.pt")
    torch.save(hmodels64, HERE + "/models_heads_fp64.pt")

    # ---- MACE through the reference's own MACEStack / blocks / symmetric_contraction / cg / irreps_tools (e3nn restated) ----
    mace = install_mace_stubs()
    gen3 = torch.Generator().manual_seed(97531)
    mmodels = {}
    heads_mace = {"graph": [{"type": "branch-0", "architecture": {"num_sharedlayers": 2, "dim_sharedlayers": 5, "num_headlayers": 2,
                                                                   "dim_headlayers": [10, 6]}}],
                  "node": [{"type": "branch-0", "architecture": {"num_headlayers": 2, "dim_headlayers": [12, 12], "type": "mlp"}}]}
    for name, (max_ell, node_max_ell, corr, layers, hidden) in {"mace_l2_nu2": (2, 1, 2, 2, 8), "mace_l2_nu3": (2, 2, 3, 3, 4),
                                                                "mace_l3_nu2": (3, 2, 2, 2, 4), "mace_one_layer": (2, 1, 2, 1, 8)}.items():
        b = toy_batch(gen3, [7, 9, 5], 3.5, input_dim=1)
        b.y = torch.randn(b.x.shape[0], 1, generator=gen3)
        torch.manual_seed(0)
        m = mace.MACEStack("node_attributes, equiv_node_feat, inv_node_feat, edge_attributes, edge_features, edge_index",
                           "node_attributes, edge_attributes, edge_features, edge_index", 6.0, "bessel", None, 8, None,
                           max_ell, node_max_ell, 10.0, 5, corr, 1, hidden, [1, 3], 0, "", "", 0, ["graph", "node"], heads_mace,
                           "relu", "mae", None, loss_weights=[1.0, 1.0], freeze_conv=False, initial_bias=None,
                           num_conv_layers=layers, num_nodes=9, graph_pooling="mean")
        m.eval()
        state = {k: v.clone() for k, v in m.state_dict().items()}
        inp = t2d(b)
        pos0 = b.pos.clone().requires_grad_(True)
        b.pos = pos0
        pred = m(b)
        obj = pred[0].sum() + pred[1].pow(2).sum()
        forces = torch.autograd.grad(obj, pos0, retain_graph=True)[0]
        grads = torch.autograd.grad(obj, list(m.parameters()), allow_unused=True)
        mmodels[name] = {"state": state, "inputs": inp, "pred": [p.detach() for p in pred], "dobj_dpos": forces.detach(),
                         "grads": {n: (g.detach() if g is not None else None) for (n, _), g in zip(m.named_parameters(), grads)},
                         "cfg": dict(max_ell=max_ell, node_max_ell=node_max_ell, correlation=corr, num_conv_layers=layers, hidden_dim=hidden)}
    torch.save(mmodels, HERE + "/models_mace.pt")
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()
