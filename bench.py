#!/usr/bin/env python
"""bench.py - edges/sec of the Equiformer graph-attention hot path (fwd+bwd training step) on B200.

Contract (one JSON line on stdout from rank 0):
    python bench.py --gpus N --steps K --warmup W                    # sm_100a kernels behind the drop-in modules
    python bench.py --impl reference --gpus N --steps K --warmup W   # the oracle restatement on the host cores (CPU arm)
    python bench.py --impl reference-gpu ...                         # the same reference-style op chain, eager torch on the B200
    python bench.py ... --dump-outputs DIR    # also write the last timed step's loss / gradients / parameters as DIR/*.npy

Workloads (``--workload``; BASELINE.json ``configs``):
    qm9      [1] (default, the config the metric is quoted on) 128 molecules x ~18 atoms, radius 5 A, Lmax=2,
             ``graph_attention_transformer_nonlinear_l2``; step = forward + L1 loss + backward (+ all-reduce) + AdamW
    md17_l3  [2] 5 aspirin-sized conformers, ``graph_attention_transformer_nonlinear_exp_l3_md17``; step = energy + autograd
             forces + L2-MAE loss (weights 1 / 100, scripts/train/md17/equiformer/se_l3/target@aspirin.sh:22-23) + double
             backward + AdamW
    oc20_l1  [3] 16 periodic frames x ~73 atoms x ~50 neighbours per GPU, ``l1_256_nonlinear`` (IS2RE), energy L1 loss
    stress   [4] one periodic cell of 10 000 atoms, ~50 neighbours (E ~ 5e5), Lmax=2 model of [1]; replicas under --gpus N

* ``value``    - edges/s with the step's inputs already resident in HBM when the timed region starts.
* ``e2e``      - the same step from pinned HOST tensors: H2D copy of the inputs and D2H read of the loss inside the timed
                 region, every step.  ``--stream K`` (qm9): K >= 16 DIFFERENT seeded batches cycle through the step
                 (``graphs.BucketedForwardBackward``: a few captured graphs over size buckets) - reported as ``e2e``.
* ``roofline`` - the dominant hand-written kernel family by summed device time (CUDA events around every launch of our
                 kernels in an instrumented eager pass): algorithmic bytes / time against the measured HBM copy bandwidth
                 AND, for contraction kernels, useful flops / time against the TF32 tensor roof (half the measured bf16
                 throughput of MEASURED_PEAKS.json) - both are reported, ``bound`` names the nearer one.
* ``cpu_baseline`` - the oracle (reference-style op chain, torch CPU) on a bounded sample of the same workload (N = 1 only).

Multi-GPU: one process per GPU (torchrun), independent batch per rank (weak scaling), NCCL all-reduce of one flat gradient
bucket per step; time = max over ranks, measured with CUDA events between barriers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC_QM9 = "edges/sec fwd+bwd, QM9 Lmax=2 batch"
WORKLOADS = {
    "qm9": dict(metric=METRIC_QM9, model="graph_attention_transformer_nonlinear_l2", n_graphs=128,
                text="QM9 synthetic batch: 128 molecules x ~18 atoms, radius 5 A, Lmax=2 "
                     "(graph_attention_transformer_nonlinear_l2), fwd+bwd+AdamW"),
    "md17_l3": dict(metric="edges/sec fwd+bwd (energy+force step), MD17 aspirin Lmax=3",
                    model="graph_attention_transformer_nonlinear_exp_l3_md17", n_graphs=5,
                    text="MD17 aspirin-like: 5 conformers x 21 atoms, radius 5 A, Lmax=3 (se_l3), energy + autograd forces, "
                         "L2-MAE loss (weights 1 / 100), double backward + AdamW"),
    "oc20_l1": dict(metric="edges/sec fwd+bwd, OC20 IS2RE l1_256_nonlinear frames", model="graph_attention_transformer_oc20",
                    n_graphs=16, text="OC20 IS2RE synthetic frames: 16 periodic frames x ~73 atoms x ~50 neighbours per GPU, "
                                      "l1_256_nonlinear, fwd+bwd+AdamW"),
    "stress": dict(metric="edges/sec fwd+bwd, 10k-atom periodic cell Lmax=2", model="graph_attention_transformer_nonlinear_l2",
                   n_graphs=1, text="stress: one periodic cell of 10 000 atoms, ~50 neighbours within 5 A (E ~ 5e5), Lmax=2, "
                                    "fwd+bwd+AdamW; one independent cell per GPU"),
}


# --------------------------------------------------------------------------------------------------- synthetic inputs


def make_inputs(workload: str, seed: int, n_graphs=None):
    """Host tensors of one step of the workload (seeded)."""
    from equiformer_b200 import synthetic as S
    g = torch.Generator().manual_seed(seed + 1000)
    if workload == "qm9":
        n = n_graphs or 128
        pos, batch, z = S.qm9_like_batch(n, seed=seed)
        return dict(pos=pos, batch=batch, z=z, target=torch.randn(n, 1, generator=g))
    if workload == "md17_l3":
        n = n_graphs or 5
        confs = [S.aspirin_like(seed=seed * 16 + s) for s in range(n)]
        pos = torch.cat([c[0] for c in confs])
        z = torch.cat([c[2] for c in confs])
        batch = torch.cat([torch.full((21,), i, dtype=torch.long) for i in range(n)])
        return dict(pos=pos, batch=batch, z=z, target=torch.randn(n, 1, generator=g), ftarget=torch.randn(21 * n, 3, generator=g))
    if workload == "oc20_l1":
        n = n_graphs or 16
        pos, batch, z, tags, cell = S.oc20_like_frames(n, seed=seed)
        return dict(pos=pos, batch=batch, z=z, tags=tags, cell=torch.diag_embed(cell[:, None].expand(-1, 3)).float(),
                    target=torch.randn(n, 1, generator=g))
    if workload == "stress":
        pos, batch, z, side = S.stress_cell(n_graphs or 10000, seed=seed)
        return dict(pos=pos, batch=batch, z=z, cell=(torch.eye(3) * side).view(1, 3, 3).float(), target=torch.randn(1, 1, generator=g))
    raise ValueError(workload)


def count_edges(workload: str, inp) -> int:
    from equiformer_b200.graph import radius_graph, radius_graph_pbc
    if workload in ("oc20_l1", "stress"):
        return int(radius_graph_pbc(inp["pos"], inp["batch"], inp["cell"], 5.0, 500)[0].shape[1])
    return int(radius_graph(inp["pos"], 5.0, inp["batch"], max_num_neighbors=1000).shape[1])


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self._stop_evt = threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([f.strip() for f in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx.append(float(s[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    """(HBM GB/s, TF32 dense TFLOP/s, source).  TF32 tensor roof = half the measured dense bf16 throughput."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]) / 2.0, "measured (MEASURED_PEAKS.json: hbm_gbs, bf16_tflops / 2)"
    return 6650.0, 1125.0, "fallback (B200_PROFILING.md: 6.65 TB/s, 2.25 PFLOP/s bf16 / 2)"


def dump_outputs(out_dir: str, arrays, max_elems: int = 1 << 22):
    """Write each array as ``<out_dir>/<name>.npy``, flattened.  An array of more than ``max_elems`` elements is replaced
    by a fixed, seeded sample of that many of its elements, so two builds' dumps compare position for position and the
    three arrays of a step stay well under 64 MB."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.reshape(-1)
        if t.numel() > max_elems:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:max_elems].sort().values
            t = t[idx]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def ncu_traffic(kernel: str):
    """dram bytes per launch of the dominant kernel from the committed ncu summary (profiles/), if present."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                return json.load(f).get(kernel)
        except Exception:
            return None
    return None


# --------------------------------------------------------------------------------------------------- reference arms


def oracle_setup(workload: str, n_sample: int, seed: int, device="cpu"):
    """Oracle parameters (the mirror's state_dict, fp32) + a bounded sample of the workload + the step closure."""
    from equiformer_b200.nets import model_entrypoint
    from equiformer_b200.nets.graph_attention_transformer_oc20 import OC20_L1_256_NONLINEAR
    from oracle import equiformer_ref as R
    torch.manual_seed(0)
    if workload in ("qm9", "stress"):
        model = model_entrypoint(WORKLOADS[workload]["model"])(irreps_in="5x0e", radius=5.0, num_basis=128)
        cfg = R.Config()
    elif workload == "md17_l3":
        model = model_entrypoint(WORKLOADS[workload]["model"])(irreps_in="64x0e", radius=5.0, num_basis=32)
        cfg = R.Config(irreps_node_embedding="128x0e+64x1e+64x2e+32x3e", irreps_sh="1x0e+1x1e+1x2e+1x3e",
                       irreps_head="32x0e+16x1e+16x2e+8x3e", irreps_mlp_mid="384x0e+192x1e+192x2e+96x3e",
                       basis_type="exp", number_of_basis=32, max_atom_type=64, qm9_atom_remap=False)
    else:
        model = model_entrypoint("graph_attention_transformer_oc20")(**OC20_L1_256_NONLINEAR)
        cfg = R.Config(irreps_node_embedding="256x0e+128x1e", irreps_sh="1x0e+1x1e", irreps_head="32x0e+16x1e",
                       irreps_mlp_mid="768x0e+384x1e", num_heads=8, max_atom_type=84, qm9_atom_remap=False,
                       avg_degree=23.395238876342773, avg_num_nodes=77.81317)
    params = {k: v.to(device).requires_grad_(v.is_floating_point() and v.numel() > 0)
              for k, v in R.cast_params(model.state_dict(), torch.float32).items()}
    inp = make_inputs(workload, seed, n_graphs=n_sample)
    n_graphs = int(inp["target"].shape[0])
    edges = count_edges(workload, inp)
    cell_offsets = None
    if workload in ("oc20_l1", "stress"):
        from equiformer_b200.graph import radius_graph_pbc
        edge, cell_offsets, _ = radius_graph_pbc(inp["pos"], inp["batch"], inp["cell"], 5.0, 500)
        inp["src"], inp["dst"], inp["cell_offsets"] = edge[0], edge[1], cell_offsets
    inp = {k: v.to(device) for k, v in inp.items()}

    def step():
        for v in params.values():
            if v.is_floating_point():
                v.grad = None
        if workload == "md17_l3":
            e, f = R.energy_and_forces(params, cfg, inp["pos"], inp["batch"], inp["z"], n_graphs, create_graph=True)
            loss = (e - inp["target"]).norm(dim=-1).mean() + 100.0 * (f - inp["ftarget"]).norm(dim=-1).mean()
        elif workload == "oc20_l1":
            out = R.model_forward_oc20(params, cfg, inp["pos"], inp["cell"], inp["batch"], inp["z"], inp["tags"], n_graphs,
                                       inp["src"], inp["dst"], inp["cell_offsets"])
            loss = (out - inp["target"]).abs().mean()
        elif workload == "stress":
            raise RuntimeError("the oracle has no periodic QM9-model entry; use the qm9 sample as the CPU baseline of 'stress'")
        else:
            out = R.model_forward(params, cfg, inp["pos"], inp["batch"], inp["z"], n_graphs)
            loss = (out - inp["target"]).abs().mean()
        loss.backward()
        return float(loss.detach())

    return step, edges, n_graphs


def host_threads() -> int:
    """Threads for the CPU arm: one per physical core of ONE socket (torchrun pins OMP_NUM_THREADS=1; one thread per
    logical core oversubscribes the oracle's small matmuls by two orders of magnitude, and threads spread over two sockets
    made the same arm vary 3.8x between boxes in round 1)."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:
        n = None
    if not n:
        n = max(1, (os.cpu_count() or 2) // 2)
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    return max(1, min(n, 32))


def pin_one_socket(n: int):
    """Restrict this process to the first ``n`` distinct physical cores (lowest core ids = one socket); returns the ids."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
        seen, cpus = set(), []
        for c in allowed:
            try:
                with open(f"/sys/devices/system/cpu/cpu{c}/topology/core_id") as f:
                    core = int(f.read())
                with open(f"/sys/devices/system/cpu/cpu{c}/topology/physical_package_id") as f:
                    pkg = int(f.read())
            except OSError:
                core, pkg = c, 0
            if pkg == 0 and (pkg, core) not in seen:
                seen.add((pkg, core))
                cpus.append(c)
            if len(cpus) == n:
                break
        if cpus:
            os.sched_setaffinity(0, set(cpus))
        return cpus
    except (AttributeError, OSError):
        return []


def reference_sample(workload: str, requested: int) -> int:
    if requested:
        return requested
    return {"qm9": 32, "md17_l3": 5, "oc20_l1": 2, "stress": 32}[workload]


def run_reference(args):
    """The reference's CPU path stand-in: oracle op chain on the cores of one socket, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    base = "qm9" if wl == "stress" else wl
    gpu = args.impl == "reference-gpu"
    threads = host_threads()
    cpus = [] if gpu else pin_one_socket(threads)
    torch.set_num_threads(threads)
    if gpu:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    n_sample = reference_sample(wl, args.ref_graphs) if not gpu else (args.ref_graphs or WORKLOADS[base]["n_graphs"])
    step, edges, n_graphs = oracle_setup(base, n_sample, 0, device="cuda" if gpu else "cpu")
    sync = torch.cuda.synchronize if gpu else (lambda: None)
    for _ in range(args.warmup):
        step()
    sync()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    sync()
    dt = (time.perf_counter() - t0) / args.steps
    value = edges / dt
    full = WORKLOADS[base]["n_graphs"]
    where = "eager torch CUDA ops on the B200 (allow_tf32 off)" if gpu else "torch CPU fp32"
    sample = f"{n_graphs} of the {full} graphs ({edges} edges) per step, oracle op chain fwd+bwd, {where}"
    line = {"impl": args.impl, "metric": WORKLOADS[wl]["metric"], "value": value, "unit": "edges/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOADS[wl]["text"], "sample": sample, "cpu_affinity": cpus,
                       "same_config": n_graphs == full},
            "cpu_baseline": {"value": value, "unit": "edges/s", "cores": 0 if gpu else threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------- our arm


def build_model(workload: str, dev, alpha_drop: float):
    from equiformer_b200.nets import model_entrypoint
    from equiformer_b200.nets.graph_attention_transformer_oc20 import OC20_L1_256_NONLINEAR
    torch.manual_seed(0)
    name = WORKLOADS[workload]["model"]
    if workload == "md17_l3":
        model = model_entrypoint(name)(irreps_in="64x0e", radius=5.0, num_basis=32)
    elif workload == "oc20_l1":
        model = model_entrypoint(name)(**OC20_L1_256_NONLINEAR)
    else:
        model = model_entrypoint(name)(irreps_in="5x0e", radius=5.0, num_basis=128)
    model = model.to(dev).train()
    for m in model.modules():        # attention-weight dropout is the only stochastic op of the step
        if isinstance(m, torch.nn.Dropout):
            m.p = alpha_drop
    return model


def run_ours(args):
    import torch.distributed as dist
    from equiformer_b200 import _lib, ops
    from equiformer_b200.graph import radius_graph_pbc
    from equiformer_b200.graphs import BucketedForwardBackward, GraphedForwardBackward, GraphedStep
    from equiformer_b200.parallel import FlatAdamW, FlatGradAllReduce, broadcast_parameters, init_distributed

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the edge path has no CPU implementation "
                           "(use --impl reference for the CPU oracle)")
    if not _lib.LIB_PATH.exists():
        _lib.build()
    wl = args.workload
    rank, local, world = init_distributed("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.backends.cuda.matmul.allow_tf32 = False  # fp32 parity: the reference trains with --no-amp
    torch.backends.cudnn.allow_tf32 = False

    model = build_model(wl, dev, args.alpha_drop)
    broadcast_parameters(model)
    bucket = FlatGradAllReduce(model.parameters())
    lr, wd = {"qm9": (5e-4, 5e-3), "md17_l3": (2e-4, 1e-6), "oc20_l1": (2e-4, 1e-3), "stress": (5e-4, 5e-3)}[wl]
    opt = FlatAdamW(model.named_parameters(), bucket, lr=lr, weight_decay=wd, no_decay=model.no_weight_decay())

    n_stream = max(args.stream, 1)
    hosts = []
    for i in range(n_stream):      # independent inputs per rank (weak scaling) and, with --stream, per step
        inp = make_inputs(wl, seed=rank * 1000 + i)
        hosts.append({k: v.pin_memory() for k, v in inp.items()})
    keys = [k for k in hosts[0]]
    edges_of = [count_edges(wl, h) for h in hosts]
    edges_local = sum(edges_of) / len(edges_of)
    dev_in = {k: v.to(dev) for k, v in hosts[0].items()}
    h2d_bytes = sum(t.numel() * t.element_size() for t in hosts[0].values())

    l1 = lambda out, tgt: (out - tgt).abs().mean()
    l2mae = lambda pred, tgt: (pred - tgt).norm(p=2, dim=-1).mean()

    def pbc_graph(d):
        edge, offs, _ = radius_graph_pbc(d["pos"], d["batch"], d["cell"], 5.0, 500)
        src, dst = edge[0], edge[1]
        offsets = torch.bmm(offs.to(d["pos"].dtype).view(-1, 1, 3), d["cell"].index_select(0, d["batch"].index_select(0, dst))).view(-1, 3)
        edge_vec = d["pos"].index_select(0, src) - d["pos"].index_select(0, dst) + offsets
        return src, dst, edge_vec

    def forward_loss(d):
        if wl == "qm9":
            out = model(f_in=None, pos=d["pos"], batch=d["batch"], node_atom=d["z"], n_graphs=d["target"].shape[0])
            return l1(out, d["target"])
        if wl == "md17_l3":
            energy, forces = model(node_atom=d["z"], pos=d["pos"], batch=d["batch"])
            return 1.0 * l2mae(energy, d["target"]) + 100.0 * l2mae(forces, d["ftarget"])
        src, dst, edge_vec = pbc_graph(d)
        if wl == "oc20_l1":
            out = model.forward_edges(edge_vec, d["batch"], d["z"], d["tags"], src, dst, n_graphs=d["target"].shape[0])
        else:
            out = model.forward_edges(d["pos"], d["batch"], d["z"], src, dst, n_graphs=1, edges_sorted=True, edge_vec=edge_vec)
        return l1(out, d["target"])

    def step_eager(d):
        bucket.zero_grad()
        loss = forward_loss(d)
        loss.backward()
        bucket.reduce()
        opt.step()
        return loss

    graphed = None
    use_graph = args.graph
    if use_graph:
        if wl == "qm9":
            cls = BucketedForwardBackward if args.stream > 1 else GraphedForwardBackward
            graphed = cls(model, l1, bucket, max_radius=5.0)
        elif wl == "md17_l3":
            # the whole energy + force step - a backward inside the forward and the backward of that - in one CUDA graph
            def captured_md17(pos, target, ftarget, batch, z, src, dst, row_ptr):
                csr = ops.Graph.__new__(ops.Graph)
                csr.n_nodes, csr.n_edges, csr.perm = int(batch.shape[0]), int(src.numel()), None
                csr.src, csr.dst, csr.row_ptr = src, dst, row_ptr
                csr._src_perm = csr._src_row_ptr = None
                p = pos.detach().requires_grad_(True)
                energy, forces = model.forward_edges(z, p, batch, src, dst, graph=csr, n_graphs=target.shape[0])
                return 1.0 * l2mae(energy, target) + 100.0 * l2mae(forces, ftarget)
            graphed = GraphedStep(captured_md17, bucket)
        else:
            def captured(edge_vec, pos, target, batch, z, tags, src, dst, row_ptr):
                csr = ops.Graph.__new__(ops.Graph)
                csr.n_nodes, csr.n_edges, csr.perm = int(batch.shape[0]), int(src.numel()), None
                csr.src, csr.dst, csr.row_ptr = src, dst, row_ptr
                csr._src_perm = csr._src_row_ptr = None
                if wl == "oc20_l1":
                    out = model.forward_edges(edge_vec, batch, z, tags, src, dst, graph=csr, n_graphs=target.shape[0])
                else:
                    out = model.forward_edges(pos, batch, z, src, dst, graph=csr, n_graphs=1, edge_vec=edge_vec)
                return l1(out, target)
            graphed = GraphedStep(captured, bucket)

    def step_graph(d):
        if wl == "qm9":
            loss = graphed(d["pos"], d["batch"], d["z"], d["target"])     # neighbour search (eager) + replay
        elif wl == "md17_l3":
            from equiformer_b200.graph import radius_graph_csr
            edge, row_ptr = radius_graph_csr(d["pos"], 5.0, d["batch"], max_num_neighbors=1000)
            loss = graphed((int(d["pos"].shape[0]), int(edge.shape[1]), int(d["target"].shape[0])),
                           [d["pos"], d["target"], d["ftarget"], d["batch"], d["z"], edge[0], edge[1], row_ptr])
        else:
            src, dst, edge_vec = pbc_graph(d)                             # periodic neighbour list (eager) + replay
            n = d["batch"].shape[0]
            counts = torch.zeros(n, dtype=torch.int64, device=dev).index_add_(0, dst, torch.ones_like(dst))
            row_ptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
            torch.cumsum(counts, 0, out=row_ptr[1:])
            tags = d.get("tags", d["z"])
            loss = graphed((n, int(src.numel()), int(d["target"].shape[0])),
                           [edge_vec, d["pos"], d["target"], d["batch"], d["z"], tags, src, dst, row_ptr])
        bucket.reduce()
        opt.step()
        return loss

    step = step_graph if use_graph else step_eager

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n_steps, from_host, profile, fn=None, stream=False):
        fn = fn or step
        barrier()
        ops.PROFILE = profile
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        last = None
        for i in range(n_steps):
            if from_host:
                h = hosts[i % len(hosts)] if stream else hosts[0]
                d = {k: v.to(dev, non_blocking=True) for k, v in h.items()}
                last = fn(d).item()            # D2H read of the loss every step
            else:
                last = fn(dev_in)
        end.record()
        barrier()
        ops.PROFILE = None
        ms = torch.tensor([start.elapsed_time(end)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / n_steps, last

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_eager(dev_in)
    torch.cuda.synchronize()
    mem_gb = torch.cuda.max_memory_allocated(dev) / 1e9
    if use_graph:
        for i in range(warm if args.stream <= 1 else len(hosts)):      # includes the one-off captures
            step({k: v.to(dev) for k, v in hosts[i % len(hosts)].items()} if args.stream > 1 else dev_in)
        torch.cuda.synchronize()

    # per-kernel CUDA-event timing needs eager launches (events cannot be read back from inside a graph replay):
    # an instrumented eager pass of the same step gives the roofline numbers, the headline is timed on `step`.
    profile = ops.KernelProfile(time_events=True, presleep_cycles=200_000)   # ~0.1 ms GPU-side head start per timed launch
    ms_eager, _ = timed(min(args.steps, 5) if wl != "qm9" else args.steps, from_host=False, profile=profile, fn=step_eager)
    n_prof_steps = min(args.steps, 5) if wl != "qm9" else args.steps
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    mark = os.environ.get("EQF_BENCH_CUDA_PROFILER") == "1"   # `ncu --profile-from-start off`: launches of the headline region
    if mark:
        torch.cuda.cudart().cudaProfilerStart()
    if use_graph:
        ms_step, last_step_loss = timed(args.steps, from_host=False, profile=None)
    else:
        ms_step, last_step_loss = timed(args.steps, from_host=False, profile=None, fn=step_eager)
    if mark:
        torch.cuda.cudart().cudaProfilerStop()
    clocks = sampler.stop() if sampler else None
    # what the last timed step handed back (the loss) and left behind (its averaged gradients, the parameters after its
    # AdamW update), copied before the e2e pass below trains on; float32, as the step computes them
    last_step = ({"loss": last_step_loss.detach().float().cpu(), "grad": bucket.flat.float().cpu(),
                  "params": opt.flat.float().cpu()} if args.dump_outputs else None)
    ms_e2e, last_loss = timed(args.steps if args.stream <= 1 else max(args.steps, len(hosts)), from_host=True, profile=None,
                              stream=args.stream > 1)

    edges_total = torch.tensor([edges_of[0]], device=dev, dtype=torch.float64)
    edges_stream = torch.tensor([edges_local], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(edges_total)
        dist.all_reduce(edges_stream)
    edges_total, edges_stream = edges_total.item(), edges_stream.item()

    if rank == 0:
        hbm_peak, tf32_peak, peak_src = measured_peaks()
        summ = profile.summary()
        own = {k: v for k, v in summ.items() if not k.startswith("gemm_fast_f32")}
        dominant = max(own, key=lambda k: own[k]["ms"]) if own else None
        kernels = {}
        for name, d in summ.items():
            kernels[name] = {"launches_per_step": d["launches"] / n_prof_steps, "ms_per_step": d["ms"] / n_prof_steps,
                             "gb_s": d["bytes"] / (d["ms"] * 1e-3) / 1e9 if d["ms"] > 0 else None,
                             "tflops_useful": d["flops"] / (d["ms"] * 1e-3) / 1e12 if d["ms"] > 0 and d["flops"] else None}
        roof = None
        if dominant:
            d = summ[dominant]
            gbs = d["bytes"] / (d["ms"] * 1e-3) / 1e9
            tfs = d["flops"] / (d["ms"] * 1e-3) / 1e12
            f_hbm, f_tensor = gbs / hbm_peak, tfs / tf32_peak
            bound = "tensor" if f_tensor > f_hbm else "hbm"
            def entry(k):
                g = own[k]["bytes"] / (own[k]["ms"] * 1e-3) / 1e9
                t = own[k]["flops"] / (own[k]["ms"] * 1e-3) / 1e12
                return {"gb_s": g, "frac_hbm": g / hbm_peak, "tflops_useful": t, "frac_tensor_tf32": t / tf32_peak,
                        "ms_per_step": own[k]["ms"] / n_prof_steps}
            roof = {"kernel": dominant, "bound": bound,
                    "achieved": tfs if bound == "tensor" else gbs, "peak": tf32_peak if bound == "tensor" else hbm_peak,
                    "unit": "TFLOP/s" if bound == "tensor" else "GB/s", "frac": f_tensor if bound == "tensor" else f_hbm,
                    "hbm": {"achieved": gbs, "peak": hbm_peak, "frac": f_hbm, "unit": "GB/s"},
                    "tensor": {"achieved_useful": tfs, "peak_tf32_dense": tf32_peak, "frac": f_tensor, "unit": "TFLOP/s",
                               "note": "useful fp32 flops; the 3xTF32 scheme issues 3 tensor-core products per useful one"},
                    "traffic": ncu_traffic(dominant), "peak_source": peak_src,
                    "bytes_per_launch": d["bytes"] / d["launches"], "us_per_launch": d["ms"] * 1e3 / d["launches"],
                    "share_of_step": d["ms"] / (ms_step * n_prof_steps), "launches_per_step": d["launches"] / n_prof_steps,
                    "runner_up": {k: entry(k) for k in sorted(own, key=lambda k: -own[k]["ms"])[1:4]},
                    "timed_in": "instrumented eager pass of the same step: CUDA events around each launch of our kernels, "
                                "a GPU-side delay queued before each pair keeps host launch gaps out of the interval"}
        cpu = None
        if not args.no_cpu_baseline and world == 1:      # the CPU leg is an N = 1 figure (rank 0's host cores)
            base = "qm9" if wl == "stress" else wl
            threads = host_threads()
            cpus = pin_one_socket(threads)
            torch.set_num_threads(threads)
            n_sample = reference_sample(wl, args.ref_graphs)
            cstep, cedges, cgraphs = oracle_setup(base, n_sample, 0)
            cstep()
            t0 = time.perf_counter()
            reps = 0
            while reps < 1 or time.perf_counter() - t0 < 10.0:
                cstep()
                reps += 1
                if time.perf_counter() - t0 > 30.0:
                    break
            dt = (time.perf_counter() - t0) / reps
            cpu = {"value": cedges / dt, "unit": "edges/s", "cores": threads, "kind": "port", "affinity": cpus,
                   "sample": f"{cgraphs} of the {WORKLOADS[base]['n_graphs']} graphs ({cedges} edges) of '{base}', oracle op chain "
                             f"fwd+bwd x{reps}, torch CPU fp32"}
        line = {
            "metric": WORKLOADS[wl]["metric"], "value": edges_total / (ms_step * 1e-3), "unit": "edges/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOADS[wl]["text"], "edges_per_step": edges_total, "atoms_per_rank": int(hosts[0]["pos"].shape[0]),
                       "parallelism": f"dp{world}", "l2": f"inputs larger than L2: {mem_gb:.2f} GB of activations per step",
                       "dropout": (f"attention-weight dropout p = {args.alpha_drop} (reference default 0.2; the only stochastic op "
                                   "of the step; p = 0 keeps the run comparable with the parity tests)"),
                       "fused": (f"EQF_FUSED={ops._FUSED_MODE}: the depth-wise tensor product is produced on chip as the A operand of "
                                 f"the tcgen05 GEMMs (K1) from {ops._FUSED_MIN_EDGES} edges per call in 'auto' mode - "
                                 + ("ON" if ops._FUSED and (ops._FUSED_MODE == "1" or edges_of[0] >= ops._FUSED_MIN_EDGES) else "OFF")
                                 + " for this workload"),
                       "gemm": ("tcgen05 3xTF32, hand-written (forward / dgrad from "
                                f"{ops._GEMM_MIN_M} rows, wgrad from {ops._WGRAD_MIN_K} reduction rows); below "
                                "that the grouped warp-MMA 3xTF32 kernel (all degrees of a linear per launch); no cuBLAS on the path")
                               if ops.gemm_backend() == "tf32x3" else ops.gemm_backend(),
                       "launch": ("CUDA-graph replay of forward+loss+backward; neighbour search, all-reduce and AdamW eager"
                                  + (f"; stream of {len(hosts)} different batches over {graphed.captures} captured size buckets"
                                     if args.stream > 1 and graphed is not None else "")) if use_graph else "eager",
                       "eager_ms_per_step": ms_eager},
            "e2e": {"value": (edges_stream if args.stream > 1 else edges_total) / (ms_e2e * 1e-3), "unit": "edges/s",
                    "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "distinct_batches": len(hosts), "captures": getattr(graphed, "captures", None)},
            "gpu_launches": profile.launches // max(n_prof_steps, 1),   # our kernels launched per step (instrumented pass)
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "kernels": kernels,
            "loss": last_loss, "grad_bucket_bytes": bucket.nbytes,
        }
        print(json.dumps(line), flush=True)
        if last_step is not None:
            dump_outputs(args.dump_outputs, last_step)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--workload", default="qm9", choices=sorted(WORKLOADS))
    ap.add_argument("--stream", type=int, default=0, help="qm9: cycle this many DIFFERENT seeded batches through the step (e2e)")
    ap.add_argument("--alpha-drop", type=float, default=0.0, help="attention-weight dropout probability (reference: 0.2)")
    ap.add_argument("--ref-graphs", type=int, default=0, help="graphs in the bounded CPU sample (0: per-workload default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--graph", dest="graph", action="store_true", default=True)
    ap.add_argument("--no-graph", dest="graph", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last one's loss, gradients and updated parameters as DIR/<name>.npy")
    args = ap.parse_args()
    if args.stream > 1 and args.workload != "qm9":
        ap.error("--stream is implemented for the qm9 workload")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs is implemented for --impl ours")
    if args.impl in ("reference", "reference-gpu"):
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
