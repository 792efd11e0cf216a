"""CPU tests: host-side logic, the C-ABI surface (load + exported symbols, no compute calls), and the
world_size-2 data-parallel plumbing over gloo."""
import os
import re
import subprocess
import sys

import pytest
import torch

import hydragnn_b200 as hb
from hydragnn_b200 import _lib, ops
from hydragnn_b200.synthetic import ARCH, make_samples
from test_oracle_golden import GPS_KW, HEAD_KW, MODEL_KW, PNAEQ_KW

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_library_loads_and_exports_every_declared_symbol():
    protos = _lib.prototypes()
    assert len(protos) >= 35
    src = open(_lib.HEADER).read()
    declared = set(re.findall(r"\b(hgb_\w+)\s*\(", re.sub(r"/\*.*?\*/", "", src, flags=re.S)))
    assert declared == set(protos), declared ^ set(protos)
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    L = _lib.lib()
    for name in protos:
        assert hasattr(L, name), name
    assert L.hgb_version() >= 100
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (hgb_\w+)", out))
    assert set(protos) <= exported
    # every signature in the header is plain C: no torch / C++ types
    for name, (ret, args) in protos.items():
        for t, _ in args:
            assert re.fullmatch(r"(const )?(void|float|double|int32_t|int64_t|uint64_t|int|hgb_stream_t)\*?", t), (name, t)


def test_ops_refuse_cpu_tensors_no_fallback():
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.raw_gather(torch.zeros(3, 2), torch.zeros(2, dtype=torch.int32))
    m = hb.create_model(**MODEL_KW["painn_graph_mean"])
    g = torch.load(os.path.join(ROOT, "tests/golden/models.pt"))["painn_graph_mean"]
    with pytest.raises(RuntimeError):
        m(hb.Batch(**g["inputs"]))


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libhgb.so")
    with pytest.raises(RuntimeError, match="no CPU"):
        _lib.lib()


def test_create_model_reproduces_reference_initialisation(golden_dir):
    g = torch.load(golden_dir + "/models.pt")
    for name, kw in MODEL_KW.items():
        sd = hb.create_model(use_gpu=False, **kw).state_dict()
        assert list(sd.keys()) == list(g[name]["state"].keys()), name
        for k, v in sd.items():
            assert torch.equal(v, g[name]["state"][k]), (name, k)


def test_pnaeq_initialisation_matches_reference(golden_dir):
    g = torch.load(golden_dir + "/models_pnaeq.pt")
    for name, c in g.items():
        sd = hb.create_model(use_gpu=False, **dict(PNAEQ_KW, graph_pooling=name.split("_")[-1], pna_deg=c["deg"])).state_dict()
        assert list(sd.keys()) == list(c["state"].keys())
        for k, v in sd.items():
            assert torch.equal(v, c["state"][k]), (name, k)
    with pytest.raises(AssertionError, match="degree"):
        hb.create_model(**dict(PNAEQ_KW, pna_deg=None))


def test_gps_initialisation_matches_reference(golden_dir):
    g = torch.load(golden_dir + "/models_gps.pt")
    for name, c in g.items():
        sd = hb.create_model(use_gpu=False, **GPS_KW[name]).state_dict()
        assert list(sd.keys()) == list(c["state"].keys())
        for k, v in sd.items():
            assert torch.equal(v, c["state"][k]), (name, k)
    with pytest.raises(ValueError):
        hb.create_model(**dict(GPS_KW["gps_egnn"], global_attn_type="performer"))


def test_mace_initialisation_matches_oracle_and_tables_agree():
    """No reference-generated golden exists for MACE (e3nn is not installable): the engine's construction order / RNG
    consumption is pinned to the oracle's restatement, and the engine's coupling tables to the oracle's."""
    from oracle import e3 as oe3, mace as omace
    from hydragnn_b200 import e3 as pe3
    from test_oracle_mace import MACE_KW
    for extra in ({}, {"max_ell": 3, "node_max_ell": 2, "correlation": 3, "hidden_dim": 4, "num_conv_layers": 3}):
        kw = dict(MACE_KW, **extra)
        torch.manual_seed(0)
        so = omace.MACEOracle(**kw).state_dict()
        se = hb.create_model(mpnn_type="MACE", use_gpu=False, **kw).state_dict()
        assert list(so.keys()) == list(se.keys())
        for k in so:
            assert so[k].shape == se[k].shape and torch.allclose(so[k].float(), se[k].float(), atol=1e-6), k
    g = torch.load(os.path.join(ROOT, "tests/golden/models_mace.pt"))          # produced by the reference's own MACE files
    for name, c in g.items():
        se = hb.create_model(mpnn_type="MACE", use_gpu=False, **dict(MACE_KW, **c["cfg"])).state_dict()
        assert list(se.keys()) == list(c["state"].keys()), name
        for k, v in se.items():
            assert v.shape == c["state"][k].shape and torch.allclose(v, c["state"][k], atol=1e-6), (name, k)
    for a in [(1, 1, 0), (1, 2, 3), (2, 2, 2), (3, 2, 1), (3, 3, 2)]:
        assert torch.allclose(pe3.w3j(*a), oe3.wigner_3j(*a), atol=1e-14)
    coupling = oe3.Irreps("1x0e+1x1o+1x2e")
    for l, nu in [(0, 1), (0, 2), (1, 2), (0, 3), (1, 3), (2, 2)]:
        assert torch.allclose(pe3.u_matrix(2, l, nu), omace.u_matrix_real(coupling, "%d%s" % (l, "eo"[l % 2]), nu), atol=1e-12)
    v = torch.randn(20, 3, dtype=torch.float64)
    assert torch.allclose(pe3.spherical_harmonics_cl(3, torch.nn.functional.normalize(v, dim=-1)), oe3.spherical_harmonics(3, v), atol=1e-12)
    assert pe3.tp_paths(1, 2, 2) == [(0, 0, 0), (1, 1, 0), (0, 1, 1), (1, 0, 1), (1, 2, 1), (0, 2, 2), (1, 1, 2)]
    with pytest.raises(AssertionError, match="max_ell"):
        hb.create_model(mpnn_type="MACE", use_gpu=False, **dict(MACE_KW, max_ell=None))


def test_node_head_variants_initialisation_matches_reference(golden_dir):
    g = torch.load(golden_dir + "/models_heads.pt")
    for name, kw in HEAD_KW.items():
        sd = hb.create_model(use_gpu=False, **kw).state_dict()
        assert list(sd.keys()) == list(g[name]["state"].keys()), name
        for k, v in sd.items():
            assert torch.equal(v, g[name]["state"][k]), (name, k)
    with pytest.raises(AssertionError, match="num_nodes"):
        hb.create_model(use_gpu=False, **dict(HEAD_KW["egnn_mlp_per_node"], num_nodes=None))


def test_create_model_errors_mirror_reference():
    with pytest.raises(ValueError, match="Unknown mpnn_type"):
        hb.create_model(**dict(MODEL_KW["egnn_mlip"], mpnn_type="GIN"))
    with pytest.raises(ValueError, match="Inconsistent number of loss weights"):
        hb.create_model(**dict(MODEL_KW["egnn_mlip"], task_weights=[1.0, 1.0]))
    with pytest.raises(ValueError, match="Unsupported graph_pooling"):
        hb.create_model(**dict(MODEL_KW["egnn_mlip"], graph_pooling="median"))
    m = hb.create_model(**ARCH["md17_egnn"])
    assert m.num_heads == 1 and m.head_type == ["node"] and m.energy_weight == 1.0 and m.graph_pooling == "mean"
    assert str(m.model) == "EGCLStack"


def test_create_model_config_surface():
    cfg = {"Architecture": dict(ARCH["qm9_painn"], freeze_conv_layers=False, initial_bias=None, num_nodes=9, edge_dim=None,
                                equivariance=None, pe_dim=0, global_attn_engine=None),
           "Training": {"loss_function_type": "mse", "precision": "bf16"}}
    m = hb.create_model_config(cfg)
    assert m.precision == "bf16" and str(m) == "Base" and type(m).__name__ == "PAINNStack"
    cfg["Training"]["precision"] = "fp64"
    with pytest.raises(ValueError):
        hb.create_model_config(cfg)


def test_data_batch_container():
    a = hb.Data(x=torch.ones(2, 1), pos=torch.zeros(2, 3), edge_index=torch.tensor([[0], [1]]), y=torch.ones(1, 1), energy=torch.tensor(1.0))
    b = hb.Data(x=torch.ones(3, 1), pos=torch.zeros(3, 3), edge_index=torch.tensor([[0, 2], [1, 0]]), y=torch.ones(1, 1), energy=torch.tensor(2.0))
    bt = hb.Batch.from_data_list([a, b])
    assert bt.num_graphs == 2 and bt.num_nodes == 5 and bt.edge_index.tolist() == [[0, 2, 4], [1, 3, 2]]
    assert bt.batch.tolist() == [0, 0, 1, 1, 1] and bt.energy.tolist() == [1.0, 2.0] and bt.edge_shifts is None
    assert "x" in bt and "edge_attr" not in bt and dict(bt.items())["y"].shape == (2, 1)
    c = bt.clone()
    c.x += 1
    assert float(bt.x.sum()) == 5.0 and bt["x"] is bt.x
    assert not hasattr(bt, "dataset_name")


def test_head_indices_and_precision():
    m = hb.create_model(**MODEL_KW["egnn_equiv_multihead"])
    d = hb.Batch(y=torch.zeros(100, 1), batch=torch.tensor([0, 0, 1, 1, 1]), y_loc=torch.tensor([[0, 1, 7], [0, 1, 10]]))
    d._num_graphs = 2
    hi = hb.get_head_indices(m, d)
    assert hi[0].tolist() == [0, 7] and hi[1].tolist() == list(range(1, 7)) + list(range(8, 17))
    from hydragnn_b200.train import resolve_precision
    assert resolve_precision("bfloat16")[0] == "bf16" and resolve_precision(None)[0] == "fp32"
    with pytest.raises(ValueError):
        resolve_precision("fp64")
    with pytest.raises(ValueError):
        resolve_precision("int8")


def test_flat_adamw_views_share_storage():
    m = hb.create_model(**MODEL_KW["painn_graph_mean"])
    before = {k: v.clone() for k, v in m.state_dict().items()}
    opt = hb.FlatAdamW(m, lr=1e-3)
    for k, v in m.state_dict().items():
        assert torch.equal(v, before[k])
    n = sum(p.numel() for p in m.parameters())
    assert opt.flat_p.numel() == n
    p0 = next(m.parameters())
    opt.flat_p[:p0.numel()] = 7.0
    assert float(p0.min()) == 7.0                              # parameters are views of the flat buffer
    for p in m.parameters():
        p.grad = torch.full_like(p, 2.0)
    list(m.parameters())[3].grad = None                        # an unused parameter contributes zeros
    flat = opt.gather_grads()
    k3 = list(m.parameters())[3].numel()
    assert float(flat.sum()) == 2.0 * (n - k3)


def test_flat_adamw_is_a_torch_optimizer_and_speaks_adamw_checkpoints(monkeypatch):
    """ADVICE r1: ReduceLROnPlateau must accept it (train_validate_test.py:452-476 steps the scheduler), and optimizer
    checkpoints must move between torch.optim.AdamW (the reference, optimizer.py:12-40) and the engine in both directions."""
    from hydragnn_b200 import ops

    def cpu_adamw(p, g, m, v, step_dev, lr, b1, b2, eps, wd, gscale=1.0, hyper_dev=None):    # CPU stand-in for the CUDA kernel
        if hyper_dev is not None:
            lr, gscale = float(hyper_dev[0]), float(hyper_dev[1])
        step_dev += 1
        t = float(step_dev)
        g = g * gscale
        p.mul_(1 - lr * wd); m.mul_(b1).add_(g, alpha=1 - b1); v.mul_(b2).addcmul_(g, g, value=1 - b2)
        p.addcdiv_(m / (1 - b1 ** t), (v / (1 - b2 ** t)).sqrt() + eps, value=-lr)

    monkeypatch.setattr(ops, "adamw_step", cpu_adamw)
    kw = dict(MODEL_KW["painn_graph_mean"], use_gpu=False)
    a, b = hb.create_model(**kw), hb.create_model(**kw)
    oa, ob = hb.FlatAdamW(a, lr=1e-2), torch.optim.AdamW(b.parameters(), lr=1e-2, weight_decay=1e-2)
    assert isinstance(oa, torch.optim.Optimizer)
    sched = torch.optim.lr_scheduler.ReduceLROnPlateau(oa, mode="min", factor=0.5, patience=0)
    gen = torch.Generator().manual_seed(0)
    for it in range(3):
        for p, q in zip(a.parameters(), b.parameters()):
            p.grad = torch.randn(p.shape, generator=gen)
            q.grad = p.grad.clone()
        oa.gather_grads()
        oa.step()
        ob.step()
    for p, q in zip(a.parameters(), b.parameters()):
        torch.testing.assert_close(p, q, rtol=1e-5, atol=1e-7)
    # torch -> engine -> torch round trip of the optimizer state
    c = hb.create_model(**kw)
    oc = hb.FlatAdamW(c, lr=1.0)
    oc.load_state_dict(ob.state_dict())
    assert oc.lr == 1e-2 and float(oc.step_dev) == 3.0
    torch.testing.assert_close(oc.m, oa.m, rtol=1e-5, atol=1e-7)
    d = hb.create_model(**kw)
    od = torch.optim.AdamW(d.parameters(), lr=5.0)
    od.load_state_dict(oa.state_dict())
    assert od.param_groups[0]["lr"] == 1e-2
    s0 = od.state[next(iter(d.parameters()))]
    torch.testing.assert_close(s0["exp_avg"], ob.state[next(iter(b.parameters()))]["exp_avg"], rtol=1e-5, atol=1e-7)
    # the scheduler drives the lr the kernel reads (device vector)
    sched.step(1.0)
    sched.step(2.0)
    assert oa.lr == 5e-3
    oa.sync_hyper()
    assert abs(float(oa.hyper_dev[0]) - 5e-3) < 1e-9


WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
import hydragnn_b200 as hb
from hydragnn_b200 import ops, train
from hydragnn_b200.synthetic import ARCH

def torch_adamw(p, g, m, v, step_dev, lr, b1, b2, eps, wd, gscale=1.0, hyper_dev=None):   # CPU stand-in for the CUDA kernel (test only)
    if hyper_dev is not None:
        lr, gscale = float(hyper_dev[0]), float(hyper_dev[1])
    step_dev += 1
    t = float(step_dev)
    g = g * gscale
    p.mul_(1 - lr * wd); m.mul_(b1).add_(g, alpha=1 - b1); v.mul_(b2).addcmul_(g, g, value=1 - b2)
    p.addcdiv_(m / (1 - b1 ** t), (v / (1 - b2 ** t)).sqrt() + eps, value=-lr)
ops.adamw_step = torch_adamw
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
model = hb.create_model(**ARCH["qm9_painn"], use_gpu=False)
if rank == 1:
    with torch.no_grad():
        for p in model.parameters(): p.add_(1.0)           # deliberately different starting point
model = hb.get_distributed_model(model)                     # rank 0's weights everywhere
opt = hb.FlatAdamW(model, lr=1e-2)
for p in model.parameters():
    p.grad = torch.full_like(p, float(rank + 1))            # rank-dependent gradients: mean is 1.5
flat = opt.gather_grads()
dist.all_reduce(flat)
opt.step(grad_scale=1.0 / 2)
out = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
gathered = [torch.zeros_like(out) for _ in range(2)]
dist.all_gather(gathered, out)
assert torch.equal(gathered[0], gathered[1]), "ranks diverged"
if rank == 0:
    ref = hb.create_model(**ARCH["qm9_painn"], use_gpu=False)
    o2 = torch.optim.AdamW(ref.parameters(), lr=1e-2, weight_decay=1e-2)
    for p in ref.parameters(): p.grad = torch.full_like(p, 1.5)
    o2.step()
    r = torch.cat([p.detach().reshape(-1) for p in ref.parameters()])
    assert torch.allclose(out, r, rtol=1e-5, atol=1e-7), float((out - r).abs().max())
    print("OK")
dist.destroy_process_group()
'''


def test_two_rank_gloo_flat_allreduce_matches_single_process(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
    assert "OK" in outs[0]


def test_synthetic_workloads_shapes():
    b = make_samples("qm9_painn", 10)
    assert b.pos.shape == (90, 3) and b.x.shape == (90, 1) and b.num_graphs == 10 and b.ptr.tolist()[-1] == 90
    d = torch.cdist(b.pos.reshape(10, 9, 3), b.pos.reshape(10, 9, 3)) + torch.eye(9) * 10
    assert float(d.min()) >= 0.9
    assert torch.equal(make_samples("qm9_painn", 10).pos, b.pos)      # deterministic in the seed
    lj = make_samples("lj_egnn", 2)
    assert lj.cell.shape == (2, 3, 3) and bool(lj.pbc.all())


def test_generated_mace_header_is_in_sync_with_the_tables(tmp_path):
    """hgb_mace_gen.cuh is generated from hydragnn_b200/e3.py: regenerate it and compare with the committed file."""
    sys.path.insert(0, os.path.join(ROOT, "hydragnn_b200", "csrc"))
    try:
        import gen_mace
    finally:
        sys.path.pop(0)
    out = gen_mace.generate(str(tmp_path / "gen.cuh"))
    assert open(out).read() == open(os.path.join(ROOT, "hydragnn_b200", "csrc", "hgb_mace_gen.cuh")).read()


def test_bench_reference_arm_prints_the_contract_line():
    import json
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--ref-graphs", "32"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == "atoms_per_sec_training_step" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] == "port"


def test_c4_and_c5_synthetic_workloads_and_multihead_indices():
    b = make_samples("oc20_mace_80", 3)
    assert b.pos.shape == (240, 3) and b.cell.shape == (3, 3, 3) and bool(b.pbc.all())
    assert b.y.shape == (3 * 241, 1) and b.y_loc.tolist() == [[0, 1, 241]] * 3
    assert float(b.x.min()) >= 1 and float(b.x.max()) <= 83
    m = hb.create_model(use_gpu=False, **ARCH["oc20_mace"])
    assert str(m) == "MACEStack" and m.head_type == ["graph", "node"] and m.head_dims == [1, 3]
    hi = hb.get_head_indices(m, b)
    assert hi[0].tolist() == [0, 241, 482] and hi[1].numel() == 3 * 240 and int(hi[1][0]) == 1 and int(hi[1][-1]) == 722
    # energies and forces land where y_loc says
    assert torch.equal(b.y[hi[1]].reshape(240, 3), b.forces)
    p = make_samples("gfm_pnaeq_mini", 2)
    assert p.pe.shape == (80, 6) and p.pos.shape == (80, 3)
    # the full C4 / C5 workloads draw their graph sizes (SURVEY 8d): U{60..100} periodic cells, {9, 21, 80, 200} clusters
    c4 = make_samples("oc20_mace", 16)
    ns = (c4.ptr[1:] - c4.ptr[:-1])
    assert int(ns.min()) >= 60 and int(ns.max()) <= 100 and c4.cell.shape == (16, 3, 3) and c4.pos.shape[0] == int(ns.sum())
    assert torch.allclose(c4.cell[:, 0, 0].double() ** 3 * 0.05, ns.double(), rtol=1e-5)
    assert c4.y.shape[0] == 16 + 3 * int(ns.sum()) and c4.y_loc[:, 2].tolist() == (1 + 3 * ns).tolist()
    hi4 = hb.get_head_indices(m, c4)
    assert torch.equal(c4.y[hi4[1]].reshape(-1, 3), c4.forces)
    c5 = make_samples("gfm_pnaeq", 64)
    n5 = (c5.ptr[1:] - c5.ptr[:-1])
    assert set(n5.tolist()) <= {9, 21, 80, 200} and len(set(n5.tolist())) == 4 and c5.pe.shape == (int(n5.sum()), 6)
    assert torch.equal(c5.batch, torch.repeat_interleave(torch.arange(64), n5))
    kw = dict(ARCH["gfm_pnaeq_mini"], pna_deg=[0, 3, 5, 9])
    g = hb.create_model(use_gpu=False, **kw)
    assert str(g) == "Base" and type(g).__name__ == "PNAEqStack" and g.use_global_attn and len(g.graph_convs) == 3


def test_padded_batch_filler_layout():
    """host side of the capacity-padded step (hydragnn_b200/padded.py): unused graph slots get two filler atoms each, the last
    one the remainder; ptr / batch stay sorted and consistent; a batch that does not fit raises."""
    from hydragnn_b200.padded import filler_layout, supported
    bvec = torch.tensor([0, 0, 0, 1, 1, 2, 2, 2, 2])
    ptr, bfull, fill = filler_layout(bvec, 3, n_cap=20, g_cap=6)
    assert ptr.tolist() == [0, 3, 5, 9, 11, 13, 20] and fill == 11
    assert bfull.tolist() == bvec.tolist() + [3, 3, 4, 4] + [5] * 7 and bool((bfull[1:] >= bfull[:-1]).all())
    with pytest.raises(ValueError):
        filler_layout(bvec, 3, n_cap=12, g_cap=6)          # 3 unused slots need 6 filler atoms
    with pytest.raises(ValueError):
        filler_layout(bvec, 3, n_cap=20, g_cap=3)          # no filler graph
    m = hb.create_model(use_gpu=False, **ARCH["qm9_painn"])
    assert supported(m)
    kw = dict(ARCH["gfm_pnaeq_mini"], pna_deg=[0, 3, 5, 9])
    assert not supported(hb.create_model(use_gpu=False, **kw))                        # global attention: filler atoms would leak


def test_zero_padded_head_chain_is_the_same_function_on_cpu():
    """stacks._padded_chain (host logic of the tensor-core head MLPs): the reference's widths 64 -> 60 -> 20 -> 1 are rounded up to
    multiples of 32 with zero-padded weights / biases; the padded chain, sliced at the end, is the same function of the ORIGINAL
    parameters: same outputs, same gradients (the padding's gradient is dropped by F.pad's backward), for an activation with
    act(0) != 0 as well.  The decision itself needs many rows, an aligned input width and at least one odd width."""
    import torch.nn as nn
    from hydragnn_b200 import stacks

    class Rows:                      # the decision only looks at the shape of the input (and wants a CUDA tensor)
        is_cuda = True

        def __init__(self, rows, k):
            self.shape = (rows, k)

        def numel(self):
            return self.shape[0] * self.shape[1]

    torch.manual_seed(3)
    for act in (nn.ReLU, nn.Sigmoid):
        seq = nn.Sequential(nn.Linear(64, 60), act(), nn.Linear(60, 20), act(), nn.Linear(20, 1))
        mods = list(seq)
        assert stacks._padded_chain(mods, Rows(1000, 64)) is None                    # few rows: launch-bound, not worth it
        assert stacks._padded_chain(mods, Rows(200000, 60)) is None                  # input width is not a multiple of 32
        assert stacks._padded_chain(list(nn.Sequential(nn.Linear(64, 64), act(), nn.Linear(64, 32))), Rows(200000, 64)) is None
        assert stacks._padded_chain(mods + [nn.Dropout(0.1)], Rows(200000, 64)) is None   # not a plain Linear / activation chain
        padded = stacks._padded_chain(mods, Rows(200000, 64))
        assert [tuple(w.shape) for w, _ in padded] == [(64, 64), (32, 64), (32, 32)]
        assert [tuple(b.shape) for _, b in padded] == [(64,), (32,), (32,)]
        x = torch.randn(50, 64)
        want = seq(x)
        h = x
        for i, (w, b) in enumerate(padded):
            h = torch.nn.functional.linear(h, w, b)
            if i < 2:
                h = act()(h)
        got = h[:, :1]
        torch.testing.assert_close(got, want, rtol=1e-6, atol=1e-6)
        gw = torch.autograd.grad(want.square().sum(), list(seq.parameters()))
        gp = torch.autograd.grad(got.square().sum(), list(seq.parameters()))
        for a, b in zip(gp, gw):
            assert a.shape == b.shape
            torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-6)
