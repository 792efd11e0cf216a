#!/usr/bin/env python
"""bench.py -- atoms/sec of a full training step on synthetic radius-graph batches (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 5                     # engine arm, one B200, config C2 (QM9-shape PaiNN)
    python bench.py --workload md17_egnn|oc20_mace|gfm_pnaeq|lj_egnn   # the other BASELINE.json configs (SURVEY 8d C3/C4/C5/C1)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1     # CPU arm (oracle on the host cores)
    python bench.py --steps 20 --warmup 5 --dump-outputs DIR           # + what the last timed step computed, as DIR/<name>.npy

One "step" = neighbour build (radius graph, periodic for C1/C4, + CSR plans) -> forward -> loss -> backward -> flat gradient
all-reduce -> fused AdamW on one batch.  Weak scaling: every rank owns ``--graphs`` graphs per step; ``value`` = atoms processed
by all ranks / max-over-ranks device time.  Prints ONE JSON line on rank 0.

Timing design (VERDICT r1 "weak" #1): every step is bracketed by its own CUDA event on every rank; the timed region runs
``--regions`` (3) times and the MEDIAN region is the reported one (all regions are listed); per-step median / p90 / max and the
slowest rank are printed; the clock sampler reads NVML in-process and is started BEFORE the warm-up, so nothing forks or
initialises NVML inside a timed window; with N > 1 the NCCL all-reduce is captured INSIDE the step's CUDA graph, so a step is one
replay with no host round-trip.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

# workload -> defaults and SURVEY 8(d) roofline constants (forward algorithmic bytes per atom, training-step multiplier)
WL = {
    "qm9_painn": dict(cfg="C2", graphs=16384, precision="bf16", fwd_bytes=5536, mult=3, ref_graphs=1024,
                      desc="PaiNN F=64 L=2 R=5, 9-atom graphs r=7 k=5, graph energy head, MSE, AdamW"),
    "md17_egnn": dict(cfg="C3", graphs=8192, precision="fp32", fwd_bytes=9696, mult=6, ref_graphs=512,
                      desc="EGNN F=64 L=3, 21-atom graphs r=7 k=5, node energy head, E + E/atom + F (autograd forces, double backward), MSE, AdamW"),
    "oc20_mace": dict(cfg="C4", graphs=256, precision="bf16", fwd_bytes=62400, mult=3, ref_graphs=8,
                      desc="MACE F=64 max_ell=2 node_max_ell=1 nu=2 R=8 L=2, periodic cells of U{60..100} atoms at 0.05/A^3, r=6 all neighbours "
                           "(~45/atom), graph energy + node forces heads, MAE, AdamW"),
    "gfm_pnaeq": dict(cfg="C5", graphs=128, precision="fp32", fwd_bytes=88000 + 3 * 4 * 64 * 4, mult=3, ref_graphs=16,
                      desc="PNAEq F=64 L=3 R=6 + GPS multihead attention (8 heads, pe_dim 6), graph sizes drawn from {9,21,80,200}, r=5 k=20, "
                           "graph energy + node forces heads, MAE, AdamW"),
    "lj_egnn": dict(cfg="C1", graphs=4096, precision="fp32", fwd_bytes=3392, mult=6, ref_graphs=256,
                    desc="EGNN F=32 L=2, periodic 27-atom LJ cells r=5 k=5, node energy head, E + E/atom + F, MSE, AdamW"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="qm9_painn", choices=sorted(WL))
    ap.add_argument("--graphs", type=int, default=None, help="graphs per GPU per step (default: the workload's saturating batch)")
    ap.add_argument("--nbatches", type=int, default=4, help="distinct pre-generated batches cycled through")
    ap.add_argument("--regions", type=int, default=3, help="how many times the timed region of --steps steps is run (median reported)")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-capture-allreduce", action="store_true", help="keep the NCCL all-reduce outside the step graph (two replays per step)")
    ap.add_argument("--ref-graphs", type=int, default=None, help="graphs per step of the CPU arm / cpu_baseline sample")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-kernel-shares", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, per-task losses, head predictions, flat "
                         "gradient, parameters after the update) as DIR/<name>.npy in float32 (rank 0)")
    ap.add_argument("--precision", default=None, choices=["bf16", "fp32"],
                    help="bf16 = tensor-core (tcgen05, TF32-in/fp32-acc) Linears; fp32 = exact SIMT kernels; default: the config's")
    a = ap.parse_args()
    w = WL[a.workload]
    a.graphs = a.graphs or w["graphs"]
    a.ref_graphs = a.ref_graphs or w["ref_graphs"]
    a.precision = a.precision or w["precision"]
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", 1451.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1451.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / power / throttle reasons sampled DURING the timed regions -- in-process NVML on a thread that is started
    (and has initialised NVML) before the warm-up; only samples taken inside [mark_begin, mark_end] windows are reported."""

    def __init__(self, index):
        self.index, self.rows, self.windows, self._stop, self.err = index, [], [], threading.Event(), None
        self.th = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.th = threading.Thread(target=self._run, daemon=True)
            self.th.start()
        except Exception as ex:  # pragma: no cover
            self.err = repr(ex)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), sm, pw, rs))
            except Exception as ex:  # pragma: no cover
                self.err = repr(ex)
                return
            time.sleep(0.004)

    def mark_begin(self):
        self._t0 = time.perf_counter()

    def mark_end(self):
        self.windows.append((self._t0, time.perf_counter()))

    def stop(self):
        if self.th is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: %s" % self.err]}
        time.sleep(0.05)
        self._stop.set()
        self.th.join(timeout=1.0)
        nv = self.nv
        inside = [r for r in self.rows if any(a <= r[0] <= b for a, b in self.windows)] or self.rows
        sm = sorted(r[1] for r in inside)
        bits = 0
        for r in inside:
            bits |= r[3]
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, v in names.items() if bits & v)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm, "reasons": reasons, "samples": len(inside),
                "power_w_max": max((r[2] for r in inside), default=None), "source": "in-process NVML, 4 ms period, timed windows only"}


# -----------------------------------------------------------------------------------------------------------
# CPU arm: the oracle's training step on the host cores
# -----------------------------------------------------------------------------------------------------------
def cpu_step_rate(workload, graphs, steps, warmup, verbose_threads=True):
    """atoms/s of the pure-torch oracle (same model, same batch shape, fp32, best host thread count).  The radius graph
    is built once outside the timed steps, as the reference does at preprocessing."""
    import oracle
    from oracle.workloads import add_edges_cpu, arch_for, make_samples
    batch = add_edges_cpu(make_samples(workload, graphs, seed=4321), workload)
    kw = arch_for(workload, batch)
    model = oracle.base.create_model(**kw)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    mlip = kw.get("enable_interatomic_potential", False)
    import hydragnn_b200 as hb
    hi = None if mlip else hb.get_head_indices(model, batch)

    def step():
        opt.zero_grad()
        if mlip:
            batch.pos.requires_grad_(True)
            loss, _ = model.energy_force_loss(model(batch), batch)
        else:
            loss, _ = model.loss(model(batch), batch.y, hi)
        loss.backward()
        opt.step()
        return float(loss)

    # "all the host threads it can use": ATen's intra-op pool does not scale to 128 threads on these small
    # tensors, so time one step at several pool sizes and keep the fastest (reported as `cores`; every timing is printed).
    ncpu = os.cpu_count() or 1
    best, per_threads = None, {}
    for nt in sorted({ncpu, max(1, ncpu // 2), 32, 16, 8}):
        if nt > ncpu:
            continue
        torch.set_num_threads(nt)
        step()
        t0 = time.perf_counter()
        step()
        d1 = time.perf_counter() - t0
        per_threads[str(nt)] = round(d1 * 1e3, 2)
        if best is None or d1 < best[0]:
            best = (d1, nt)
    torch.set_num_threads(best[1])
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    atoms = batch.pos.shape[0]
    return atoms / dt, dt, atoms, torch.get_num_threads(), per_threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WL[args.workload]
    rate, dt, atoms, threads, per_threads = cpu_step_rate(args.workload, args.ref_graphs, args.steps, max(args.warmup, 1))
    sample = "%d graphs (%d atoms) per step, %d steps; edges prebuilt as the reference does at preprocessing" % (
        args.ref_graphs, atoms, args.steps)
    line = {"impl": "reference", "metric": "atoms_per_sec_training_step", "value": rate, "unit": "atoms/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s (%s): %s" % (args.workload, w["cfg"], w["desc"]), "graphs_per_step": args.ref_graphs,
                       "note": "pure-torch oracle restating the reference's PyG path (PyG is not installable here); per-atom rate of a bounded "
                               "sample of the same workload (--ref-graphs sets the sample; the engine arm's batch is %d graphs)" % w["graphs"],
                       "ms_per_step_by_threads": per_threads},
            "cpu_baseline": {"value": rate, "unit": "atoms/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "atoms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# -----------------------------------------------------------------------------------------------------------
# per-entry-point algorithmic bytes (fp32 storage), used for the roofline of the dominant kernel
# -----------------------------------------------------------------------------------------------------------
def _alg_flops(entry, a, ctx):
    """ALGORITHMIC flops of the entries that are tensor- / FMA-bound rather than HBM-bound (None otherwise)."""
    if entry == "hgb_mha_tc_fwd":             # S = Q K^T and O = P V over ONE dense sequence of n tokens: 2 n^2 f each
        return 4.0 * a["n"] * a["n"] * a["f"]
    if entry == "hgb_mha_tc_bwd":             # S again, dP = dO V^T, dV = P^T dO, dQ = dS K, dK = dS^T Q
        return 10.0 * a["n"] * a["n"] * a["f"]
    if entry in ("hgb_egnn_edge_fwd", "hgb_egnn_edge_bwd_data", "hgb_egnn_edge_wgrad"):
        return 2.0 * ctx["E"] * a["h"] * a["h"]
    return None


def _alg_bytes(entry, a, ctx):
    """ALGORITHMIC bytes of one C-ABI call (DESIGN.md section 4 lists every formula).  ``a``: argument dict by header name."""
    N, E = ctx["N"], ctx["E"]
    nz = lambda k: 1 if a.get(k) else 0  # noqa: E731
    if entry == "hgb_tc_linear":
        return 4 * a["m"] * (a["k_red"] + a["n_out"] * (1 + nz("z") + nz("addend") + nz("gsrc")))
    if entry == "hgb_tc_wgrad":
        return 4 * a["m"] * (a["n_out"] + a["k_out"])
    if entry in ("hgb_gemm",):
        return 4 * (a["m"] * a["k"] + a["k"] * a["n"] + a["m"] * a["n"])
    if entry in ("hgb_linear_fwd", "hgb_linear_smallk_fwd"):
        return 4 * a["m"] * (a["k"] + a["n"] * (1 + nz("z")))
    if entry == "hgb_linear_smallk_bwd":
        return 4 * a["m"] * (a["n"] * (1 + nz("y") + nz("z")) + a["k"] * (1 + nz("dx")))
    if entry == "hgb_gather_rows":
        return 4 * (a["e"] * a["c"] + a["e"]) + 4 * min(a["e"], N) * a["c"]
    if entry == "hgb_segment_sum":
        rows = E if a["n"] >= N else N
        return 4 * (rows * a["c"] + rows + a["n"] * a["c"])
    if entry == "hgb_painn_message_fwd":
        return a["n"] * 11 * a["f"] * 4 + E * 64 + (a["n"] + 1) * 4
    if entry == "hgb_painn_message_bwd":
        return a["n"] * 14 * a["f"] * 4 + E * 64 + (E * 48 if a.get("g_epack") else 0)
    if entry in ("hgb_painn_update_pre_fwd",):
        return 4 * a["n"] * a["f"] * (3 + 1 + 2)
    if entry == "hgb_painn_update_post_fwd":
        return 4 * a["n"] * a["f"] * (3 + 6 + 1 + 3 + 1 + 3)
    if entry == "hgb_painn_update_post_bwd_a":
        return 4 * a["n"] * a["f"] * (1 + 3 + 6 + 3)
    if entry == "hgb_painn_update_bwd":
        return 4 * a["n"] * a["f"] * (1 + 3 + 2 + 3 + 6 + 2 + 6 + 1)
    if entry == "hgb_act_bwd":
        return 4 * a["count"] * 3
    if entry == "hgb_adamw_step":
        return 4 * a["count"] * 7
    if entry == "hgb_egnn_edge_fwd":          # per edge: Q[col] row gathered + s, nbr, perm + the two mask words; per node: PQ read, sums written
        return E * (4 * a["h"] + 28) + a["n"] * 3 * a["h"] * 4
    if entry in ("hgb_egnn_edge_bwd_data", "hgb_egnn_edge_wgrad"):    # per edge: gz1 written (bwd) / Q[col] gathered (wgrad) + masks, s, perm
        return E * (4 * a["h"] + 28) + a["n"] * 2 * a["h"] * 4
    if entry == "hgb_mace_tp_scatter_fwd":
        return None
    return None


# -----------------------------------------------------------------------------------------------------------
# engine arm
# -----------------------------------------------------------------------------------------------------------
def run_engine(args):
    import hydragnn_b200 as hb
    from hydragnn_b200 import _lib, ops, radius
    from hydragnn_b200.synthetic import ARCH, WORKLOADS, make_samples

    ws = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()                                    # NVML is initialised here, long before any timed window
    if ws > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl, w = WL[args.workload], WORKLOADS[args.workload]
    G = args.graphs
    pbc = bool(w.get("pbc") or w.get("pbc_box"))
    gps = bool(w.get("pe_dim"))

    # ---- host batches (pinned) and their static device twins ------------------------------------------------
    in_keys = ["x", "pos", "y", "energy", "forces", "pe"]
    host, devb = [], []
    for b in range(args.nbatches):
        cpu = make_samples(args.workload, G, seed=1234 + 1000 * rank + b)
        keys = [k for k in in_keys if getattr(cpu, k) is not None]
        hb_ = {k: cpu[k].pin_memory() for k in keys}
        host.append(hb_)
        d = hb.Batch(**{k: torch.empty_like(v, device=dev) for k, v in hb_.items()})
        d.batch, d.ptr, d._num_graphs = cpu.batch.to(dev), cpu.ptr.to(dev).int(), G     # topology of the batch: resident
        if pbc:
            d.cell, d.pbc = cpu.cell.to(dev).double().contiguous(), cpu.pbc.to(dev).int().contiguous()
            d._cutoff = torch.full((G,), float(w["radius"]), dtype=torch.float64, device=dev)
        if getattr(cpu, "y_loc", None) is not None:
            d.y_loc = cpu.y_loc
        for k in keys:
            d[k].copy_(hb_[k])
        devb.append(d)
    n_atoms = [int(d.pos.shape[0]) for d in devb]
    h2d_bytes = sum(v.numel() * v.element_size() for v in host[0].values())

    def build_edges(d, known=None):
        """the neighbour build of one resident batch (rows a1 / a2); `known` = sizes promised by the warm-up run"""
        if pbc:
            ei, _, sh, deg, outptr, c = radius.radius_graph_pbc(d.pos.detach(), d.cell, d.pbc, d._cutoff, d.ptr, G, w["max_neighbours"],
                                                                known=known)
            d.edge_index, d.edge_shifts = ei, sh
            d._hgb_col_sorted = (ei, outptr, d.ptr)
            sizes = (c, int(ei.shape[1]))
        else:
            ei, rowptr = radius.radius_graph(d.pos.detach(), w["radius"], d.ptr, G, False, w["max_neighbours"],
                                             known_e=None if known is None else known[1])
            d.edge_index = ei
            d._hgb_col_sorted = (ei, rowptr, d.ptr)           # what hb.get_radius_graph(...)(d) records: edges grouped by target / graph
            sizes = (0, int(ei.shape[1]))
        if gps:                                               # serialized_dataset_loader.py:186-189
            d.rel_pe = (d.pe[d.edge_index[0]] - d.pe[d.edge_index[1]]).abs()
        for k in ("_hgb_plan", "_hgb_gcsr"):                  # index plans are rebuilt every step (new edges)
            d.__dict__.pop(k, None)
        return sizes

    # ---- model: data-dependent knobs from a probe batch that is the same on every rank -------------------------
    probe = make_samples(args.workload, min(G, 64), seed=99).to(dev)
    probe._num_graphs = min(G, 64)
    probe.ptr = probe.ptr.int()
    if pbc:
        probe.cell, probe.pbc = probe.cell.double().contiguous(), probe.pbc.int().contiguous()
        probe._cutoff = torch.full((probe._num_graphs,), float(w["radius"]), dtype=torch.float64, device=dev)
    Gsave, G = G, probe._num_graphs
    build_edges(probe)
    G = Gsave
    kw = dict(ARCH[args.workload])
    pn, pe_ = probe.pos.shape[0], probe.edge_index.shape[1]
    if kw["mpnn_type"] == "MACE":
        kw["avg_num_neighbors"] = pe_ / pn
    if kw["mpnn_type"] == "PNAEq":
        kw["pna_deg"] = torch.bincount(torch.bincount(probe.edge_index[1], minlength=pn)).tolist()
    del probe
    mlip = bool(kw.get("enable_interatomic_potential", False))
    model = hb.get_distributed_model(hb.set_precision(hb.create_model(**kw), args.precision))
    opt = hb.FlatAdamW(model, lr=1e-3)
    opt.sync_hyper(1.0 / ws)
    hidx = [None if mlip else hb.get_head_indices(model, d) for d in devb]
    capture_ar = ws > 1 and not args.no_capture_allreduce

    def step(d, hi, known=None, with_opt=True, collective=True):
        """the full hot path on one resident batch"""
        build_edges(d, known)
        opt.zero_grad()
        m = model.module
        if mlip:
            d.pos.requires_grad_(True)
            pred = model(d)
            loss, tasks = m.energy_force_loss(pred, d)
        else:
            pred = model(d)
            loss, tasks = m.loss(pred, d.y, hi)
        flat = opt.backward(loss)
        if with_opt:
            if ws > 1 and collective:
                dist.all_reduce(flat)
            opt.step(1.0 / ws)
        return loss.detach(), [t.detach() for t in tasks], [p.detach() for p in pred]

    # eager warm-up (also measures the sizes per batch and the number of libhgb launches per step)
    sizes = []
    for d, hi in zip(devb, hidx):
        sizes.append(build_edges(d))
        step(d, hi)
    torch.cuda.synchronize()
    ops.check_guard(dev)
    n_edges = [s[1] for s in sizes]
    c0 = _lib.launch_count()
    step(devb[0], hidx[0], known=sizes[0])
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - c0

    use_graph = not args.no_graph
    graphs, outs, g_opt = [], [], None
    if use_graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for d, hi, sz in zip(devb, hidx, sizes):
                step(d, hi, known=sz)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        one_graph = ws == 1 or capture_ar
        for d, hi, sz in zip(devb, hidx, sizes):
            g = torch.cuda.CUDAGraph()
            with ops.capture_graph(g):
                out = step(d, hi, known=sz, with_opt=one_graph)
            graphs.append(g)
            outs.append(out)
        if not one_graph:
            g_opt = torch.cuda.CUDAGraph()
            with ops.capture_graph(g_opt):
                opt.step(1.0 / ws)

    loss_host = torch.zeros(1).pin_memory()
    # e2e: the inputs of step i+1 travel host -> device on a copy stream while step i computes (what a prefetching loader
    # does); every step still pays its own H2D copy and its own loss read-back inside the timed region.
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(args.nbatches)]      # inputs of batch b are on the device
    released = [torch.cuda.Event() for _ in range(args.nbatches)]   # the step that used batch b has been enqueued and finished
    state = {"prefetched": -1, "last": None}

    def issue_copy(i):
        b = i % args.nbatches
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(released[b])
            for k in host[b]:
                devb[b][k].detach().copy_(host[b][k], non_blocking=True)
            ready[b].record(copy_stream)
        state["prefetched"] = i

    for ev in released:
        ev.record()

    def run_step(i, e2e):
        b = i % args.nbatches
        d = devb[b]
        if e2e:
            if state["prefetched"] != i:
                issue_copy(i)
            torch.cuda.current_stream().wait_event(ready[b])
        if use_graph:
            graphs[b].replay()
            if g_opt is not None:
                dist.all_reduce(opt.flat_g)
                g_opt.replay()
            out = outs[b]
        else:
            out = step(d, hidx[b], known=sizes[b])
        state["last"] = out                     # (loss, per-task losses, predictions) of this step
        if e2e:
            released[b].record()
            loss_host.copy_(out[0].reshape(1), non_blocking=True)
            if args.nbatches > 1:
                issue_copy(i + 1)

    K, R = args.steps, max(1, args.regions)
    atoms_region = sum(n_atoms[i % args.nbatches] for i in range(K))           # atoms this rank processes in one region

    def timed(e2e, with_clocks):
        """R regions of K steps; per-step CUDA events on every rank.  -> (per-rank [R, K] step ms, region ms [R])"""
        for i in range(args.warmup):
            run_step(i, e2e)
        torch.cuda.synchronize()
        per_step = torch.zeros(R, K, dtype=torch.float64)
        region_ms = torch.zeros(R, dtype=torch.float64)
        for r in range(R):
            state["prefetched"] = -1            # the first timed step issues (and waits for) its own copy
            if ws > 1:
                dist.barrier()
            torch.cuda.synchronize()
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
            if with_clocks and sampler:
                sampler.mark_begin()
            evs[0].record()
            for i in range(K):
                run_step(i, e2e)
                evs[i + 1].record()
            torch.cuda.synchronize()
            if with_clocks and sampler:
                sampler.mark_end()
            if ws > 1:
                dist.barrier()
            for i in range(K):
                per_step[r, i] = evs[i].elapsed_time(evs[i + 1])
            region_ms[r] = evs[0].elapsed_time(evs[K])
        return per_step, region_ms

    def reduce_timing(per_step, region_ms):
        """max over ranks of every region (the contract's timing) + per-step statistics + slowest rank"""
        if ws > 1:
            allr = [torch.zeros(R, device=dev, dtype=torch.float64) for _ in range(ws)]
            dist.all_gather(allr, region_ms.to(dev))
            alls = [torch.zeros(R, K, device=dev, dtype=torch.float64) for _ in range(ws)]
            dist.all_gather(alls, per_step.to(dev))
            allr, alls = torch.stack(allr).cpu(), torch.stack(alls).cpu()            # [ws, R], [ws, R, K]
            an = torch.tensor([float(atoms_region)], device=dev, dtype=torch.float64)
            dist.all_reduce(an)
            atoms_all = float(an)
        else:
            allr, alls, atoms_all = region_ms[None], per_step[None], float(atoms_region)
        reg = allr.max(dim=0).values                                                   # [R] max over ranks
        order = sorted(range(R), key=lambda r: float(reg[r]))
        med = order[len(order) // 2]
        steps_max = alls.max(dim=0).values.reshape(-1)                                 # per-step max over ranks, all regions
        srt = sorted(steps_max.tolist())
        stats = {"regions_ms": [round(float(x), 4) for x in reg], "region_used": med,
                 "step_ms_median": round(statistics.median(srt), 4), "step_ms_p90": round(srt[min(len(srt) - 1, int(0.9 * len(srt)))], 4),
                 "step_ms_max": round(srt[-1], 4), "slowest_rank": int(allr[:, med].argmax()),
                 "rank_region_ms": [round(float(x), 4) for x in allr[:, med]]}
        return float(reg[med]) / K, atoms_all, stats

    ps, rg = timed(False, True)
    ms_dev, atoms_all, stats_dev = reduce_timing(ps, rg)
    ps, rg = timed(True, False)
    ms_e2e, _, stats_e2e = reduce_timing(ps, rg)
    torch.cuda.synchronize()
    ops.check_guard(dev)                                     # every captured neighbour build produced the promised edge count
    clocks = sampler.stop() if sampler else None
    if rank == 0 and args.dump_outputs:                      # before the profiled step below moves the parameters on
        dump_outputs(args.dump_outputs, state["last"], opt)
    value = atoms_all / K / (ms_dev * 1e-3)
    e2e = atoms_all / K / (ms_e2e * 1e-3)

    roof, shares = None, None
    if rank == 0 and not args.skip_kernel_shares:
        try:
            # rank 0 profiles one eager step on its own: no collective in it (the other ranks are not taking part)
            roof, shares = kernel_shares_and_roofline(lambda: step(devb[0], hidx[0], known=sizes[0], collective=False), _lib, args,
                                                      n_atoms[0], n_edges[0], G)
        except Exception as ex:  # pragma: no cover
            roof, shares = {"error": repr(ex)}, None
    hbm, _, src = peaks()
    step_roof = {"formula": "SURVEY 8(d): %d x %d B/atom forward" % (wl["mult"], wl["fwd_bytes"]),
                 "bytes_per_atom_step": wl["mult"] * wl["fwd_bytes"], "achieved": wl["mult"] * wl["fwd_bytes"] * (value / ws) / 1e9,
                 "peak": hbm, "unit": "GB/s", "frac": wl["mult"] * wl["fwd_bytes"] * (value / ws) / 1e9 / hbm,
                 "roofline_atoms_per_s_per_gpu": hbm * 1e9 / (wl["mult"] * wl["fwd_bytes"])}

    cpu_base = None
    if rank == 0 and ws == 1 and not args.skip_cpu_baseline:          # the CPU baseline is reported at N = 1 only
        rate, dt, atoms, threads, per_threads = cpu_step_rate(args.workload, args.ref_graphs, 3, 1)
        cpu_base = {"value": rate, "unit": "atoms/s", "cores": threads, "kind": "port",
                    "sample": "%d graphs (%d atoms) per step, 3 timed steps after 1 warm-up; edges prebuilt" % (args.ref_graphs, atoms),
                    "ms_per_step_by_threads": per_threads}

    if rank == 0:
        line = {"metric": "atoms_per_sec_training_step", "value": value, "unit": "atoms/s", "n_gpus": ws, "steps": K,
                "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "tf32" if args.precision == "bf16" else "f32", "data": "synthetic",
                "config": {"workload": "%s (%s): %s" % (args.workload, wl["cfg"], wl["desc"]),
                           "precision": "bf16 config -> fp32 parameters/activations, large-M Linears on tcgen05 kind::tf32 with fp32 "
                                        "accumulation (>= bf16 autocast of the reference)" if args.precision == "bf16" else "fp32",
                           "graphs_per_gpu": G, "atoms_per_gpu": n_atoms[0], "edges_per_gpu": n_edges[0],
                           "parallelism": "dp%d (graphs sharded by rank, one flat gradient all-reduce)" % ws,
                           "step": "neighbour build (%s) + CSR plans + fwd + loss + bwd + all-reduce + fused AdamW"
                                   % ("periodic radius graph" if pbc else "radius graph"),
                           "launch": ("cuda-graph replay per batch" + (", NCCL all-reduce captured in the step graph" if capture_ar else
                                                                       (", all-reduce between two replays" if ws > 1 else "")))
                           if use_graph else "eager",
                           "e2e_pipeline": "every step copies its inputs (%s) from pinned host memory (copy stream, issued one step "
                                           "ahead) and reads its loss back" % "/".join(host[0].keys()),
                           "l2": "%d distinct batches cycled; per-step working set (activations + saved tensors) >> 126 MB L2" % args.nbatches,
                           "timing": "%d regions of %d steps, median region reported; per-step CUDA events on every rank, max over ranks" % (R, K)},
                "timing": stats_dev, "clocks": clocks, "gpu_launches": int(launches_per_step * K),
                "e2e": {"value": e2e, "unit": "atoms/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                        "timing": stats_e2e},
                "roofline": roof, "step_roofline": step_roof, "kernel_shares": shares, "cpu_baseline": cpu_base}
        print(json.dumps(line), flush=True)
    _shutdown(ws, dev, [graphs, g_opt])


DUMP_BYTES = 64 << 20


def dump_outputs(path, out, opt):
    """Write what one training step returned to its caller (loss, per-task losses, every head's prediction) and what it left in
    the optimizer (flat gradient, parameters after the update) as float32 ``path/<name>.npy``.  An array larger than its share
    of DUMP_BYTES is replaced by a fixed, seeded sample of its elements, flattened, in index order."""
    import numpy as np
    loss, tasks, pred = out
    arrays = {"loss": loss.reshape(1), "tasks_loss": torch.stack(tasks), "grads": opt.flat_g, "params": opt.flat_p}
    arrays.update(("pred_%d" % i, p) for i, p in enumerate(pred))
    cap = DUMP_BYTES // 4 // len(arrays)
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > cap:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def _shutdown(ws, dev, keep_alive):
    """One process: drain the GPU and return, so the interpreter shuts down normally and its exit handlers run.
    Several ranks: leave without tearing NCCL down: destroying a process group whose collectives live inside captured CUDA graphs
    can block forever at interpreter exit (observed: the 2-GPU run printed its line and then hung in teardown).  Every rank drains
    its GPU, meets the others once, flushes and exits the process directly."""
    torch.cuda.synchronize()
    if ws == 1:
        return
    dist.barrier()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


def kernel_shares_and_roofline(step_fn, _lib, args, N, E, G):
    """Time share of every libhgb entry point in one eager step (CUPTI kernel durations via torch.profiler, attributed to the
    C-ABI call that launched them), and the roofline object of the DOMINANT one: achieved = its algorithmic bytes / its
    measured device time.  Measured outside the timed regions."""
    from torch.profiler import ProfilerActivity, profile
    from hydragnn_b200 import ops as _ops
    hbm, tf, src = peaks()
    # one stream for this step: with the weight-gradient kernels on their side stream two kernels share the SMs, their CUPTI
    # durations stretch and start order != launch order; per-kernel figures are of the kernel running alone, like ncu's.
    overlap, _ops.WGRAD_OVERLAP = _ops.WGRAD_OVERLAP, False
    try:
        for _ in range(2):
            step_fn()
        torch.cuda.synchronize()
        _lib.trace_begin()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step_fn()
            torch.cuda.synchronize()
        calls = _lib.trace_end()                               # [(entry, {arg: value}, n_kernel_launches)]
    finally:
        _ops.WGRAD_OVERLAP = overlap
    kern = [e for e in prof.events() if getattr(e, "device_type", None) is not None and "cuda" in str(e.device_type).lower()
            and e.name and not e.name.lower().startswith(("memcpy", "memset"))]
    kern.sort(key=lambda e: e.time_range.start)
    tot_us = sum(e.time_range.elapsed_us() for e in kern)
    is_aten = lambda n: ("at::" in n or "at_cuda" in n or "cutlass" in n or "cublas" in n.lower())  # noqa: E731
    is_lib = lambda n: ("cub::" in n or "nccl" in n.lower())  # noqa: E731
    ours = [e for e in kern if not is_aten(e.name) and not is_lib(e.name)]
    by_name = {}
    for e in kern:
        key = e.name.split("(")[0][:80]
        t = by_name.setdefault(key, [0.0, 0])
        t[0] += e.time_range.elapsed_us()
        t[1] += 1
    top_names = sorted(by_name.items(), key=lambda kv: -kv[1][0])[:12]
    shares = {"total_kernel_us": round(tot_us, 1), "libhgb_share": round(sum(e.time_range.elapsed_us() for e in ours) / max(tot_us, 1e-9), 4),
              "aten_share": round(sum(e.time_range.elapsed_us() for e in kern if is_aten(e.name)) / max(tot_us, 1e-9), 4),
              "streams": "profiled step on ONE stream (side-stream weight gradients off); the timed steps overlap them",
              "by_kernel": [{"kernel": k, "us": round(v[0], 1), "launches": v[1], "share": round(v[0] / max(tot_us, 1e-9), 4)} for k, v in top_names]}
    # attribute our kernels to the C-ABI calls in launch order
    n_expected = sum(c[2] for c in calls)
    by_entry = {}
    if n_expected == len(ours):
        pos = 0
        ctx = {"N": N, "E": E, "G": G}
        for entry, a, nl in calls:
            us = sum(e.time_range.elapsed_us() for e in ours[pos:pos + nl])
            pos += nl
            t = by_entry.setdefault(entry, {"us": 0.0, "calls": 0, "bytes": 0, "unknown": False, "flops": 0.0})
            t["us"] += us
            t["calls"] += 1
            try:
                t["flops"] += _alg_flops(entry, a, ctx) or 0.0
            except Exception:                                  # noqa: BLE001 -- a reporting extra must never break the bench line
                pass
            b = _alg_bytes(entry, a, ctx)
            if b is None:
                t["unknown"] = True
            else:
                t["bytes"] += b
        ranked = sorted(by_entry.items(), key=lambda kv: -kv[1]["us"])
        shares["by_entry"] = [{"entry": k, "us": round(v["us"], 1), "calls": v["calls"], "share": round(v["us"] / max(tot_us, 1e-9), 4),
                               "achieved_GBps": None if v["unknown"] or v["us"] == 0 else round(v["bytes"] / v["us"] * 1e-3, 1),
                               "frac_of_hbm_peak": None if v["unknown"] or v["us"] == 0 else round(v["bytes"] / v["us"] * 1e-3 / hbm, 4)}
                              for k, v in ranked[:12]]
        for row, (k, v) in zip(shares["by_entry"], ranked[:12]):
            if v["flops"] and v["us"]:
                row["achieved_TFLOPs"] = round(v["flops"] / v["us"] * 1e-6, 2)       # algorithmic flops / device time
        top, tv = ranked[0]
        ach = None if tv["unknown"] else tv["bytes"] / tv["us"] * 1e-3
        roof = {"kernel": top, "selection": "largest share of the step's GPU time (%.1f %%), CUPTI kernel durations of one eager step" %
                (100 * tv["us"] / max(tot_us, 1e-9)), "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s",
                "frac": None if ach is None else ach / hbm, "traffic": None, "peak_source": src,
                "algorithmic_bytes_per_launch": None if tv["unknown"] else tv["bytes"] / tv["calls"], "ms_per_launch": tv["us"] / tv["calls"] * 1e-3,
                "launches_per_step": tv["calls"]}
        if tv["flops"] and tv["us"]:
            tfs = tv["flops"] / tv["us"] * 1e-6
            roof["algorithmic_flops_per_launch"] = tv["flops"] / tv["calls"]
            roof["achieved_TFLOPs"] = tfs
            if top.startswith("hgb_mha_tc"):
                # attention: no [n, n] matrix in HBM, the kernel is bound by the tensor / SFU pipes.  Peak = the measured dense bf16
                # throughput / 2 (TF32 runs at half the bf16 rate); the fp32 configs issue three MMAs per product (3xTF32 split)
                roof.update({"bound": "tensor", "achieved": tfs, "peak": tf / 2, "unit": "TFLOP/s", "frac": tfs / (tf / 2),
                             "note": "algorithmic flops (4 n^2 f forward, 10 n^2 f backward); legacy mma.sync m16n8k8 TF32, 3 MMAs per product in fp32 mode"})
            else:
                roof["note"] = "SIMT fp32 FMA tile GEMMs (2 E H^2 flops): FMA-issue bound, HBM fraction reported on the algorithmic bytes"
    else:
        shares["attribution"] = "kernel count mismatch (%d traced launches vs %d profiled kernels): per-entry table skipped" % (n_expected, len(ours))
        roof = {"kernel": top_names[0][0] if top_names else None, "bound": "hbm", "achieved": None, "peak": hbm, "unit": "GB/s", "frac": None,
                "traffic": None, "peak_source": src}
    return roof, shares


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_engine(a)
