#!/usr/bin/env python
"""bench.py -- epoch seconds of the embedding-propagation hot path on N B200s (driver contract).

A "step" is one pass of the hot path over one batch: full-graph propagation through the encoder,
fused gather + BPR + L2 loss, backward through the same kernels, Adam.  ``value`` = epoch seconds =
ceil(E / batch) x mean step time with the batch's triples already in HBM; ``e2e`` = the same with the
triples arriving in pinned HOST memory every step and the two loss scalars read back (the reference's
sampler yields CPU LongTensors and its loop calls ``.item()``, model/graph/LightGCN.py:49-59).

Workloads (``--workload``; SURVEY.md section 8 shapes, synthetic power-law graphs, seed 1234):
  c5w (default)  BASELINE configs[4] weak-scaled: 1.25 M users x 0.25 M items x 125 M interactions PER GPU
                 (N = 8 is exactly the 10 M x 2 M x 1 B graph); inputs are larger than L2, no flush needed
  c4 / c3 / c2   the named Amazon-Book / Gowalla / ml-1m shapes; L2 is flushed between steps.  The default run
                 appends short legs of them under ``extra_configs`` (C4 hypergraph-diffusion, C3 HCCF, C2 LightGCN at
                 N = 1; the C4 strong-scaling point at N > 1); they go through the data facade (``data.Interaction``).

N > 1 also runs ``dist_check.parity_check`` (sharded == NCCL-only == unsharded, sharded evaluation == unsharded) on the
ranks of this very job and reports it as ``"parity"``.

``--impl reference`` times the reference's own CPU torch path (oracle/torch_path.py, the same torch calls the reference
makes, including its python sampler) on the host cores, on a bounded sample of the same workload, and prints the same JSON
line with "impl": "reference".

``--dump-outputs DIR`` writes the losses and the parameters after the last timed step of the primary workload as
``DIR/<name>.npy`` (float32, at most 64 MB; see ``dump_outputs``), so that two builds can be compared on the same inputs.
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (users, items, train interactions, batch, scales_with_gpus)
    "c5w": (1_250_000, 250_000, 125_000_000, 1_048_576, True),
    "c4": (52_000, 92_000, 3_000_000, 4096, False),
    "c3": (30_000, 41_000, 1_000_000, 4096, False),
    "c2": (6_040, 3_706, 750_000, 2048, False),
}
WORKLOAD_NOTE = {
    "c5w": "BASELINE configs[4] (10 M x 2 M x 1 B, hypergraph-diffusion encoder, row-sharded over 8 GPUs) weak-scaled: every GPU holds 1/8 of it, "
           "N = 8 is the configuration itself; the per-GPU slice is the largest shape of the list whose tables exceed L2",
    "c4": "BASELINE configs[3] (Amazon-Book shape, hypergraph-diffusion / EquivSetConv)",
    "c3": "BASELINE configs[2] (Gowalla shape; --model hccf is the HCCF + hypergraph SSL configuration)",
    "c2": "BASELINE configs[1] (ml-1m shape, LightGCN 3 layers, emb 64, 1 GPU)",
}
MODELS = {"hgnn_hd3": "HGNN_HD3 local encoder (EquivSetConv + HGCNConv), 2 layers", "lightgcn": "LightGCN, 3 layers",
          "hccf": "HCCF, 2 layers, 128 learned hyperedges, edge keep 0.8, contrastLoss on the batch's unique users/items (temp 0.2)"}
SPMM_PER_STEP = {"hgnn_hd3": 12, "lightgcn": 6, "hccf": 4}
HCCF_CONF = {"lrate": 0.001, "lr_decay": 1.0, "max_epoch": 1, "batch_size": 4096, "reg": 0.0, "embedding_size": 64, "hyper_dim": 128,
             "drop_rate": 0.2, "p": 0.5, "n_layers": 2}
HCCF_TEMP, HCCF_SS_RATE, HCCF_KEEP = 0.2, 0.1, 0.8
D = 64
REG = 0.01
LR = 0.001
# the CPU arm runs on 1 / CPU_SAMPLE_DIV of the workload (same power-law generator, same encoder, batch scaled alike)
CPU_SAMPLE_DIV = {"c5w": 8, "c4": 1, "c3": 1, "c2": 1}
EXTRA_LEGS = (("c4", "hgnn_hd3"), ("c3", "hccf"), ("c2", "lightgcn"))
PROFILE_CACHE = os.path.join(ROOT, "profiles", "kernel_counters.json")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5w", choices=sorted(WORKLOADS))
    ap.add_argument("--model", default="hgnn_hd3", choices=sorted(MODELS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_configs legs and the N > 1 parity check")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--no-clocks", action="store_true", help="diagnosis: do not poll nvidia-smi during the timed region")
    ap.add_argument("--cuda-graph", default="auto", choices=["auto", "on", "off"],
                    help="replay the training step as one CUDA graph (auto: single-GPU L2-resident workloads)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the losses and parameters of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: --impl ours only")
    return args


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def profile_counters(key):
    """Hardware counters of one launch that cannot be read outside a profiler (DRAM bytes, tensor-pipe cycles): captured once
    per shape with `tools/measure_counters.py` (ncu) and cached under profiles/kernel_counters.json, keyed by shape."""
    try:
        with open(PROFILE_CACHE) as f:
            return json.load(f).get(key)
    except (OSError, ValueError):
        return None


def spmm_algorithmic_bytes(n_rows, n_cols, nnz, d):
    """SURVEY.md section 8(d): indptr + col + val + gather + write, int64 row offsets as stored.
    Gather = the whole X once when it is L2-resident (<= 64 MB), else one row per nonzero."""
    x_bytes = 4 * d * n_cols
    gather = x_bytes if x_bytes <= 64e6 else 4 * d * nnz
    return 8 * (n_rows + 1) + 4 * nnz + 4 * nnz + gather + 4 * d * n_rows


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        note = None
        if not self.lines:  # timed region shorter than one polling period: one query right after it
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=20).stdout
                self.lines = [ln.strip() for ln in out.splitlines() if ln.strip()]
                note = "timed region shorter than the 200 ms polling period: sampled right after it"
            except (OSError, subprocess.SubprocessError):
                pass
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
               "samples": len(sm)}
        if note:
            out["note"] = note
        return out


def workload_dims(name, n_gpus):
    u, i, e, b, scales = WORKLOADS[name]
    k = n_gpus if scales else 1
    return u * k, i * k, e * k, b * k


def workload_label(workload, model_name, n_gpus):
    U, I, E, B = workload_dims(workload, n_gpus)
    return "%s: %d users x %d items x %d interactions, emb %d, %s, batch %d" % (workload, U, I, E, D, MODELS[model_name], B)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's CPU torch path on a bounded sample
# ------------------------------------------------------------------------------------------------
def cpu_reference_run(workload, model_name, steps, warmup, n_gpus):
    """The reference's training step (oracle/torch_path.py: its torch calls, its python sampler) on all host cores, on
    1 / div of the workload.  Returns the MEASURED sample step time and the scaling rule separately."""
    import numpy as np
    import torch

    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions_device
    from oracle import hgr_oracle as O
    from oracle import torch_path as T

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    U, I, E, B = workload_dims(workload, n_gpus)
    div = CPU_SAMPLE_DIV[workload] * (n_gpus if WORKLOADS[workload][4] else 1)
    su, si, se, sb = max(U // div, 64), max(I // div, 64), max(E // div, 1024), max(B // div, 256)
    t0 = time.perf_counter()
    gu, gi = powerlaw_interactions_device(su, si, se, torch.device("cpu"), seed=1234)
    train_u, train_i = gu.numpy().astype(np.int64), gi.numpy().astype(np.int64)
    csr = O.build_norm_adj(train_u, train_i, su, si)
    adj = T.coo_from_csr(*csr, (su + si, su + si))
    setup_s = time.perf_counter() - t0
    torch.manual_seed(1234)
    if model_name == "hccf":
        model = T.HCCF(adj, su, si, D, 128, 2)
        model.train()
    else:
        model = T.HGNNModel(adj, su, si, D, 2) if model_name == "hgnn_hd3" else T.LGCN(adj, su, si, D, 3)
        model.eval()  # dropout off, like the GPU arm (the reference's loop leaves it off after the first batch)
    opt = torch.optim.Adam(model.parameters(), lr=LR)
    rng = np.random.default_rng(7)
    # the reference's sampler (util/sampler.py:237-264): shuffled positives, one python-level rejection loop per sample.
    # Its dict-of-dict training sets exist before the loop starts (Interaction.__init__), so the sets of the users the
    # timed batches touch are built here, outside the timed region
    picks = [rng.integers(0, train_u.size, sb) for _ in range(warmup + steps)]
    order = np.argsort(train_u, kind="stable")
    ptr = np.zeros(su + 1, dtype=np.int64)
    np.cumsum(np.bincount(train_u, minlength=su), out=ptr[1:])
    items_by_user = train_i[order]
    sets = {}
    for pick in picks:
        for uu in np.unique(train_u[pick]).tolist():
            if uu not in sets:
                sets[uu] = set(items_by_user[ptr[uu]:ptr[uu + 1]].tolist())
    item_list = list(range(si))
    step_times, sampler_times = [], []
    for s in range(warmup + steps):
        pick = picks[s]
        t0 = time.perf_counter()
        u, p, n = T.sample_batch_pairwise(train_u[pick].tolist(), train_i[pick].tolist(), sets, item_list)
        t1 = time.perf_counter()
        if model_name == "hccf":
            T.train_step_hccf(model, opt, u, p, n, HCCF_TEMP, HCCF_SS_RATE, HCCF_KEEP)
        else:
            T.train_step(model, opt, u, p, n, REG, sb)
        t2 = time.perf_counter()
        if s >= warmup:
            sampler_times.append(t1 - t0)
            step_times.append(t2 - t0)
    step_s = sum(step_times) / len(step_times)
    steps_per_epoch = math.ceil(E / B)
    # work per step (propagation over all nonzeros + a batch of triples) is proportional to the graph: the sample holds
    # 1 / div of the interactions AND 1 / div of the batch, so one full-size step = div sampled steps
    epoch_s = step_s * div * steps_per_epoch
    sample = "%d users x %d items x %d interactions (1/%d of the workload), batch %d, %d threads, %d timed steps" % (su, si, se, div, sb, cores, steps)
    return {"epoch_s": epoch_s, "step_ms_sample": step_s * 1e3, "sampler_ms_sample": 1e3 * sum(sampler_times) / len(sampler_times),
            "cores": cores, "sample": sample, "div": div, "steps_per_epoch": steps_per_epoch, "setup_s": setup_s,
            "scaling_rule": "epoch_s = measured sample step (%.1f ms, of which the reference's python sampler %.1f ms) x %d (sample -> full graph and batch) x %d steps/epoch"
                            % (step_s * 1e3, 1e3 * sum(sampler_times) / len(sampler_times), div, steps_per_epoch),
            "nnz_per_s": 2 * se * SPMM_PER_STEP[model_name] / step_s}


def cpu_baseline_block(r):
    return {"value": r["epoch_s"], "unit": "s", "cores": r["cores"], "kind": "port", "sample": r["sample"],
            "sample_step_ms": r["step_ms_sample"], "sample_sampler_ms": r["sampler_ms_sample"], "sample_fraction": 1.0 / r["div"],
            "scaling_rule": r["scaling_rule"],
            "why_port": "the reference is a Python script tree: /root/reference does not exist on the GPU box and it has no installable package; "
                        "oracle/torch_path.py restates its torch call sequence and is pinned to its outputs by tests/test_oracle_golden.py"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.workload, args.model, args.steps, args.warmup, args.gpus)
    line = {
        "impl": "reference", "metric": "epoch_s", "value": r["epoch_s"], "unit": "s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["step_ms_sample"] * r["div"], "higher_is_better": False,
        "scaling": "weak" if WORKLOADS[args.workload][4] else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_label(args.workload, args.model, args.gpus)},
        "cpu_baseline": cpu_baseline_block(r),
        "e2e": {"value": r["epoch_s"], "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Job:
    """Process-wide state of one bench invocation (device, ranks)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit("--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run --nproc-per-node N)" % (args.gpus, self.world))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: libhgr.so has no CPU path")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        from hypergraph_diffusion_for_recommendation_b200 import _lib

        _lib.lib()

    def barrier(self):
        import torch
        import torch.distributed as dist

        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def close(self):
        import torch.distributed as dist

        if self.world > 1:
            dist.destroy_process_group()


def measure(job, workload, model_name, steps, warmup, cpu_steps, want_cpu, primary):
    """One workload on this job's GPUs; returns the JSON line (rank 0) or None."""
    import types

    import torch
    import torch.distributed as dist

    from hypergraph_diffusion_for_recommendation_b200 import _lib, encoders, ops, trainer
    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions_device

    args, world, rank, dev = job.args, job.world, job.rank, job.dev
    U, I, E, B = workload_dims(workload, world)
    small = not WORKLOADS[workload][4]
    u, i = powerlaw_interactions_device(U, I, E, dev, seed=1234)
    part, build_s, facade = None, None, None
    torch.cuda.synchronize()
    t_build = time.perf_counter()
    if world > 1:
        from hypergraph_diffusion_for_recommendation_b200 import dist as hdist

        # every rank keeps the interactions that touch the rows it owns and builds its block of the normalised adjacency
        ctx = hdist.build_partitioned(u, i, U, I, rank, world, dev)
        data, adj, part = ctx.data, ctx.adj, ctx.part
    elif small:
        # the named configurations go through the data facade the reference's models read (data.Interaction: id maps,
        # dict views, matrices from the device builder), like `SELFRec.__init__` -> `Interaction(conf, training, test)`
        from hypergraph_diffusion_for_recommendation_b200 import data as hdata

        tu, ti = heldout_pairs(u, i, U, I, dev)
        facade = hdata.Interaction(None, hdata.InteractionList(u.cpu().numpy(), i.cpu().numpy() + U),
                                   hdata.InteractionList(tu.cpu().numpy(), ti.cpu().numpy() + U), device=dev)
        data = facade
        adj = encoders._adjacency_of(data)
    else:
        # the product builder (csrc/graph_build.cu: radix sort + dedup + LUT normalisation): this is what replaces
        # Interaction.__create_sparse_bipartite_adjacency + normalize_graph_mat (data/ui_graph.py:70-84, data/graph.py:11-25)
        from hypergraph_diffusion_for_recommendation_b200 import graph as hgraph

        adj = hgraph.build_norm_adj(u, i, U, I, device=dev)
        data = types.SimpleNamespace(n_users=U, n_items=I, norm_adj=None, norm_adj_device=adj)
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t_build
    if facade is not None:
        # dense ids in order of first appearance, like the reference numbers them: the training pairs in the facade's ids
        pu, pi = facade.dense_training_pairs()
        u, i = torch.as_tensor(pu).to(dev, torch.int32), torch.as_tensor(pi).to(dev, torch.int32)
        U, I = int(facade.n_users), int(facade.n_items)
    nnz = int(adj._nnz())
    torch.manual_seed(1234)
    if model_name == "hgnn_hd3":
        model = encoders.HGNNModel(data, {"hyper_dim": D, "n_layers": 2, "p": 0.3, "drop_rate": 0.2, "batch_size": B}).to(dev)
    elif model_name == "hccf":
        if world > 1:
            raise SystemExit("--model hccf is a single-GPU workload (BASELINE configs[2])")
        model = encoders.HCCFEncoder(HCCF_CONF, data).to(dev)
    else:
        model = encoders.LGCN_Encoder(data, D, 3).to(dev)
    if model_name == "hccf":
        model.train()  # HCCF.train calls model.train() every batch (HCCF.py:81): dropout on the learned incidence stays on
    else:
        model.eval()  # dropout off: the reference's HGNN_HD3 loop calls .eval() after its first batch (HGNN_HD3.py:186-204)
    # the sharded step of an L2-resident workload is launch-bound too (~120 launches, 14 device-side barriers): captured the same
    # way (symmetric-memory barriers, multicast stores and the NCCL all_reduce are ordinary stream work): C4 at N = 2 3.60 -> 1.85
    # ms/step, N = 8 1.37 ms/step against 2.35 on one GPU.  HGR_DIST_GRAPH=0 keeps the sharded step eager.
    use_graph = small and (args.cuda_graph == "on" or (args.cuda_graph == "auto" and os.environ.get("HGR_DIST_GRAPH", "1") != "0"))
    optimizer = torch.optim.Adam(model.parameters(), lr=LR, fused=True, capturable=use_graph)

    # triples: the device sampler (csrc/sampler.cu: shuffled positives + rejection-sampled negatives, the body of
    # util/sampler.py:237-264) runs INSIDE every device-timed step; the e2e leg replays host-resident triples, the
    # interface of the reference's sampler (CPU LongTensors).  Every rank draws the same batch (same seed).
    from hypergraph_diffusion_for_recommendation_b200.sampler import PairwiseSampler

    sampler = PairwiseSampler(u, i, U, I, device=dev, seed=99)
    sgen = torch.Generator(device=dev)
    sgen.manual_seed(1234)
    perm = torch.randperm(int(u.numel()), device=dev, generator=sgen)
    n_steps = warmup + steps
    gen = torch.Generator(device=dev)
    gen.manual_seed(99)  # the same batch on every rank: the sharded step evaluates the loss on the whole batch (dist.py)
    b_local = B
    host_triples, dev_triples = [], []
    for s in range(n_steps):
        pick = torch.randint(0, int(u.numel()), (b_local,), device=dev, generator=gen)
        tu_, tp_ = u[pick].to(torch.int64), i[pick].to(torch.int64)
        tn_ = torch.randint(0, I, (b_local,), device=dev, generator=gen)
        dev_triples.append((tu_, tp_, tn_))
        host_triples.append(tuple(t.cpu().pin_memory() for t in (tu_, tp_, tn_)))
    eval_inputs = build_eval_inputs(u, i, U, I, part, rank, dev) if primary or facade is None else None
    del u, i
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if small else None

    spmm_events = []
    ops.PROFILE_EVENTS = None
    graphed = None
    if use_graph:
        # warm-up (three Adam steps on an all-zero batch, off the default stream) and capture; the timed steps then replay the
        # graph on the real batches.  The warm-up steps nudge the parameters, which timing does not depend on
        if model_name == "hccf":
            # torch.unique's variable-length result is replaced by the fixed-size sorted-with-gaps form (loss_torch.unique_padded)
            graphed = trainer.GraphedStep(lambda a, b, c: trainer.train_step_hccf(model, optimizer, a, b, c, HCCF_TEMP, HCCF_SS_RATE,
                                                                                  HCCF_KEEP, static_shapes=True), b_local, dev)
        elif world > 1:
            graphed = trainer.GraphedStep(lambda a, b, c: hdist.train_step(model, optimizer, adj, a, b, c, REG, B), b_local, dev)
        else:
            graphed = trainer.GraphedTrainStep(model, optimizer, REG, B, b_local)

    def step(tri):
        if graphed is not None:
            return graphed(tri[0], tri[1], tri[2])
        if world > 1:
            return hdist.train_step(model, optimizer, adj, tri[0], tri[1], tri[2], REG, B)
        if model_name == "hccf":
            return trainer.train_step_hccf(model, optimizer, tri[0], tri[1], tri[2], HCCF_TEMP, HCCF_SS_RATE, HCCF_KEEP)
        return trainer.train_step(model, optimizer, tri[0], tri[1], tri[2], REG, B)

    def timed(kind):
        """K steps; returns (total ms over the timed steps as max over ranks, last losses, launches)."""
        losses = None
        for s in range(warmup):
            losses = step(dev_triples[s])
            if kind == "e2e":
                losses.tolist()
        job.barrier()
        per_step = []
        launches0 = _lib.launch_count()
        ops.PROFILE_EVENTS = spmm_events if kind == "device" else None
        if world > 1 and kind == "device":  # time this rank's waits in the cross-rank barriers and its peer-store copy kernels
            adj.copy_events = []
            for pool in adj._pools.values():
                pool.wait_events = []
        t_start = torch.cuda.Event(enable_timing=True)
        t_end = torch.cuda.Event(enable_timing=True)
        if not small:
            t_start.record()
        for s in range(warmup, n_steps):
            if small:
                flush.fill_(s & 0xff)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            if kind == "e2e":
                tri = tuple(t.to(dev, non_blocking=True) for t in host_triples[s])
                losses = step(tri)
                losses.tolist()  # D2H of the step's result, like the reference's .item() calls
            else:
                off = (s * B) % max(int(perm.numel()) - B, 1)
                losses = step(sampler.batch(perm, off, min(B, int(perm.numel()))))
            if small:
                e1.record()
                per_step.append((e0, e1))
        if not small:
            t_end.record()
        job.barrier()
        ops.PROFILE_EVENTS = None
        launches = _lib.launch_count() - launches0
        if graphed is not None:  # kernels replayed from the captured graph do not pass through the library's host counter
            launches += graphed.kernels_per_replay * steps
        total = sum(a.elapsed_time(b) for a, b in per_step) if small else t_start.elapsed_time(t_end)
        if world > 1:
            t = torch.tensor([total], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total = float(t.item())
        return total, losses, launches

    clocks = ClockSampler(job.local_rank)
    if not args.no_clocks:
        clocks.start()
    if world > 1:
        adj.n_fused = adj.n_collective = adj.n_published = 0
        adj.phase_events = []
    total_ms, losses, launches = timed("device")
    clock_info = clocks.stop()
    if primary and args.dump_outputs:
        dump_outputs(args.dump_outputs, losses, model, rank, world)
    exchange = None
    if world > 1:
        # per step: propagations whose all-gather rode on the kernel epilogue (peer stores) vs NCCL collectives
        exchange = {"fused_gathers_per_step": adj.n_fused / n_steps, "nccl_gathers_per_step": adj.n_collective / n_steps,
                    "copy_kernel_gathers_per_step": adj.n_published / n_steps, "fused": bool(adj.fused),
                    "multicast": bool(getattr(adj, "multicast", False))}
        # where the sharded step spends its time on this rank (CUDA events between the phases, timed steps only)
        torch.cuda.synchronize()
        phases = {}
        for marks in adj.phase_events[warmup:]:
            for (_, e0), (name, e1) in zip(marks[:-1], marks[1:]):
                phases[name] = phases.get(name, 0.0) + e0.elapsed_time(e1) / steps
        exchange["phases_ms_rank0"] = {k: round(v, 3) for k, v in phases.items()}
        adj.phase_events = None
        waits = [e for pool in adj._pools.values() for e in (pool.wait_events or [])]
        exchange["barriers_per_step"] = len(waits) / steps
        exchange["barrier_wait_ms_per_step_rank0"] = round(sum(a.elapsed_time(b) for a, b in waits) / steps, 3)
        exchange["copy_kernel_ms_per_step_rank0"] = round(sum(a.elapsed_time(b) for a, b in adj.copy_events) / steps, 3)
        for pool in adj._pools.values():
            pool.wait_events = None
    e2e_ms, _, _ = timed("e2e")
    scale_parity = None
    if world > 1 and adj.fused and primary:
        from hypergraph_diffusion_for_recommendation_b200 import dist_check

        scale_parity = dist_check.scale_check(adj, D)
    eval_info = run_eval(job, model, eval_inputs, part, adj, workload) if eval_inputs is not None else None
    if facade is not None and not primary:
        eval_info = run_eval_facade(job, model, facade)

    ms_per_step = total_ms / steps
    steps_per_epoch = math.ceil(E / B)
    epoch_s = ms_per_step * steps_per_epoch / 1e3
    e2e_epoch_s = e2e_ms / steps * steps_per_epoch / 1e3

    # roofline of the dominant kernel (spmm_rows_async_kernel + its partial-row reduce), timed live
    torch.cuda.synchronize()
    if graphed is not None:
        # a replayed graph has no Python between its kernels to record events from: time the propagation launches of three
        # eager forward passes under the same conditions (L2 flushed); the step holds the same launches forward and backward
        ops.PROFILE_EVENTS = spmm_events
        with torch.no_grad():
            for it in range(3):
                flush.fill_(it)
                model()
        ops.PROFILE_EVENTS = None
        torch.cuda.synchronize()
    n_launch = sum(c for _, _, c in spmm_events)
    spmm_total_ms = sum(a.elapsed_time(b) for a, b, _ in spmm_events)
    avg_ms = spmm_total_ms / max(n_launch, 1)
    block = adj.block if world > 1 else adj  # the rank's block of rows when sharded
    roofline = spmm_roofline(workload, world, block, nnz, avg_ms, n_launch, ms_per_step, total_ms, graphed is not None, model_name)

    line = None
    if rank == 0:
        cpu = None
        if want_cpu:
            cpu = cpu_baseline_block(cpu_reference_run(workload, model_name, cpu_steps, 1, world))
        line = {
            "metric": "epoch_s", "value": epoch_s, "unit": "s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": False, "scaling": "weak" if WORKLOADS[workload][4] else "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_label(workload, model_name, world),
                       "baseline_config": WORKLOAD_NOTE[workload],
                       "steps_per_epoch": steps_per_epoch, "nnz": nnz,
                       "l2": "flushed between steps (256 MiB write)" if small else "inputs larger than L2 (CSR %.1f GB + tables %.2f GB)" % (nnz * 8 / 1e9, (U + I) * D * 4 / 1e9),
                       "cuda_graph": bool(use_graph), "propagation_schedule": getattr(block, "schedule", None),
                       "data_path": "data.Interaction facade" if facade is not None else "device builder on the raw pair list",
                       "parallelism": "1 GPU" if world == 1 else "row-partitioned x%d, all-gather fused into the propagation epilogue" % world},
            "e2e": {"value": e2e_epoch_s, "unit": "s", "h2d_bytes_per_step": 3 * 8 * b_local, "d2h_bytes_per_step": 8,
                    "ms_per_step": e2e_ms / steps},
            "gpu_launches": int(launches), "clocks": clock_info, "roofline": roofline, "cpu_baseline": cpu,
            "eval": eval_info, "exchange": exchange,
            "graph_build": {"seconds": build_s, "interactions": E, "nnz": nnz,
                            "what": ("this rank's block from the interactions of its own rows (dist.build_partitioned)" if world > 1 else
                                     "data.Interaction: id maps + normalised CSR on the device" if facade is not None else
                                     "device COO -> normalised CSR + split plan + work schedule (graph.build_norm_adj)")},
            "loss": [float(x) for x in losses.tolist()],
        }
        if scale_parity is not None:
            line["parity_at_scale"] = scale_parity
    del model, optimizer, sampler, adj, data, graphed, dev_triples, host_triples, eval_inputs, flush
    gc.collect()
    torch.cuda.empty_cache()
    return line


DUMP_BYTES = 60 << 20  # array data of one --dump-outputs: the files stay under 64 MB with their headers
DUMP_WHOLE_BYTES = 1 << 20  # arrays up to this size are written whole


def dump_outputs(path, losses, model, rank, world):
    """What the training step hands its caller after the last timed step: the losses it returns and the parameters it
    updated, as ``path/loss.npy`` and ``path/param.<name>.npy``.  Inputs are seeded, so two builds run with the same
    arguments can be compared file by file.  The large tables share what the small arrays leave of DUMP_BYTES and are
    written as a fixed sample of their rows (drawn with seed 0, ascending: the same rows for the same shape).  Sharded
    runs write every rank's owned rows as ``<name>.rank<r>.npy``."""
    import numpy as np
    import torch

    arrays = {"loss": losses.detach()}
    arrays.update(("param." + n, p.detach()) for n, p in model.named_parameters())
    size = {n: t.numel() * t.element_size() for n, t in arrays.items()}
    big = [n for n in arrays if size[n] > DUMP_WHOLE_BYTES]
    share = (DUMP_BYTES // world - sum(s for n, s in size.items() if n not in big)) // max(len(big), 1)
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        if name in big:
            keep = max(share // (size[name] // t.shape[0]), 1)
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows.to(t.device)]
        np.save(os.path.join(path, name + (".rank%d" % rank if world > 1 else "") + ".npy"), t.cpu().numpy())


def spmm_roofline(workload, world, block, nnz, avg_ms, n_launch, ms_per_step, total_ms, graphed, model_name):
    """The dominant kernel against the HBM roofline.  ``frac`` is the DRAM-side fraction: bytes that crossed the HBM interface
    in one launch (ncu ``dram__bytes_read.sum + dram__bytes_write.sum`` of this kernel on this shape and schedule, cached in
    profiles/kernel_counters.json by tools/measure_counters.py) / the launch time measured live / the measured copy peak.
    The SURVEY 8(d) algorithmic figure charges one 256-byte row per nonzero to HBM although L2 serves most of them; it is kept
    as ``algorithmic`` and is not a fraction of anything.  ``l2_to_sm`` compares the gathered bytes per second with the
    random-row ceiling measured on this GPU model by tools/gather_probe.py (profiles/gather_probe_r2.txt)."""
    peaks, peak_src = measured_peaks()
    peak = float(peaks["hbm_gbs"])
    n_rows, n_cols = block.shape
    alg = spmm_algorithmic_bytes(n_rows, n_cols, nnz, D)
    sched = getattr(block, "schedule", "stored")
    key = "spmm:%s:%d:%s" % (workload, world, sched)
    ctr = profile_counters(key)
    traffic = (ctr["dram_read_bytes"] + ctr["dram_write_bytes"]) if ctr else None
    sec = avg_ms * 1e-3
    have = n_launch > 0 and sec > 0
    dram_gbs = traffic / sec / 1e9 if traffic and have else None
    gathered = 4 * D * nnz  # bytes the SMs pull out of L2 for the row gathers (ncu l1tex__m_xbar2l1tex_read_bytes agrees to 1 %)
    ceiling = 18170.0       # GB/s: 250 M random 256-byte rows from an L2-resident table, profiles/gather_probe_r2.txt
    share = None
    if have:
        share = (2 * n_launch / 3 * avg_ms) / ms_per_step if graphed else (n_launch * avg_ms) / total_ms
    return {"bound": "hbm", "achieved": dram_gbs, "peak": peak, "unit": "GB/s", "frac": dram_gbs / peak if dram_gbs else None,
            "traffic": traffic, "traffic_source": (ctr or {}).get("source") if ctr else "no ncu capture cached for %s" % key,
            "kernel": "spmm_rows_async_kernel<16,4,5> (+ spmm_heavy_reduce_kernel), schedule %s" % sched,
            "launch_ms": avg_ms if have else None, "launches_timed": n_launch, "peak_source": peak_src,
            "spmm_share_of_step": share,
            "algorithmic": {"bytes": alg, "gbs": alg / sec / 1e9 if have else None,
                            "note": "SURVEY.md 8(d) formula: one 256-B row per nonzero charged to HBM; L2 serves most of them, so this is not an HBM rate"},
            "l2_to_sm": {"bytes": gathered, "gbs": gathered / sec / 1e9 if have else None, "ceiling_gbs": ceiling,
                         "frac": gathered / sec / 1e9 / ceiling if have else None,
                         "ceiling_source": "tools/gather_probe.py: pure random 256-byte row gather from a 64 MB table (profiles/gather_probe_r2.txt)"},
            "compulsory_bytes": 8 * (n_rows + 1) + 8 * nnz + 4 * D * (n_rows + n_cols),
            "note": "the kernel is bound by gather delivery (L2 -> SM, L1TEX), not by HBM: its compulsory HBM bytes take < 10 % of the launch at the "
                    "HBM peak and the DRAM-side fraction falls as the schedule improves L2 reuse (profiles/spmm_r2.md)"}


EVAL_K = 20
EVAL_MAX_USERS = 262_144  # test users ranked per GPU in the bench (all of them when the shape has fewer)


def heldout_pairs(u, i, U, I, dev):
    """Held-out interactions: fresh draws from the generator's distribution that are not training pairs (the reference's
    75 / 25 split, dataset_util.py:20-37)."""
    import torch

    from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions_device

    n_draw = max(int(u.numel()) // 3, 1024)
    tu, ti = powerlaw_interactions_device(U, I, n_draw, dev, seed=4321, cover=False, perm_seed=1234)
    key = torch.sort(u.to(torch.int64) * I + i.to(torch.int64)).values
    tkey = torch.unique(tu.to(torch.int64) * I + ti.to(torch.int64))
    tkey = tkey[~torch.isin(tkey, key)]
    return torch.div(tkey, I, rounding_mode="floor").to(torch.int32), (tkey % I).to(torch.int32)


def build_eval_inputs(u, i, U, I, part, rank, dev):
    """Training matrix rows (the mask) of the users this rank evaluates, as CSR over local user ids."""
    import torch

    u0, u1 = (0, U) if part is None else part.users_of(rank)
    n_own = min(u1 - u0, EVAL_MAX_USERS)
    m = (u >= u0) & (u < u0 + n_own)
    key = torch.sort((u[m].to(torch.int64) - u0) * I + i[m].to(torch.int64)).values
    indptr = torch.zeros(n_own + 1, dtype=torch.int64, device=dev)
    torch.cumsum(torch.bincount(torch.div(key, I, rounding_mode="floor"), minlength=n_own), 0, out=indptr[1:])
    tu, ti = heldout_pairs(u, i, U, I, dev)
    tm = (tu >= u0) & (tu < u0 + n_own)
    tkey = (tu[tm].to(torch.int64) - u0) * I + ti[tm].to(torch.int64)
    tptr = torch.zeros(n_own + 1, dtype=torch.int64, device=dev)
    torch.cumsum(torch.bincount(torch.div(tkey, I, rounding_mode="floor"), minlength=n_own), 0, out=tptr[1:])
    return {"n_own": n_own, "indptr": indptr, "indices": (key % I).to(torch.int32), "n_items": I,
            "truth_indptr": tptr.cpu().numpy(), "truth_items": (tkey % I).cpu().numpy()}


def eval_roofline(workload, world, n_users_total, n_items, ms):
    """Full-rank evaluation against the tensor roofline: the score contraction issues 3 bf16 MMAs per useful product (hi x hi,
    hi x lo, lo x hi split operands), over all item tiles in the FILTER pass and a quarter of them in the SAMPLE pass.  ``achieved`` counts the ISSUED tensor flops of the whole
    call (packing, thresholds and exact re-scoring included in the time); ``pipe_pct_elapsed`` is ncu's
    sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed of the scoring kernels (cached capture)."""
    peaks, src = measured_peaks()
    peak = float(peaks.get("bf16_tflops", 1590.0)) * world
    issued = 2.0 * D * n_items * n_users_total * 3 * 1.25  # FILTER pass over all tiles + SAMPLE pass over 1/4 of them
    tf = issued / (ms * 1e-3) / 1e12
    ctr = profile_counters("eval:%s:%d" % (workload, world)) or profile_counters("eval:%s:1" % workload)
    return {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak, "peak_source": src,
            "useful_tflops": tf / 3.75, "what": "issued bf16 MMA flops of both scoring passes / whole-call time (pack + score + threshold + exact re-score + D2H)",
            "pipe_pct_elapsed": ctr, "traffic": None}


def run_eval(job, model, ev, part, adj, workload, iters=3):
    """Full-ranking evaluation sharded by user: every rank ranks its own users against the whole item table
    (gathered once), top-EVAL_K with the training items masked.  users/s = users of all ranks / max time."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from hypergraph_diffusion_for_recommendation_b200 import evaluation as E

    world, dev = job.world, job.dev
    with torch.no_grad():
        out_u, out_i = model()[:2]
        users = torch.arange(ev["n_own"], device=dev, dtype=torch.int32)
        if world > 1:
            from hypergraph_diffusion_for_recommendation_b200 import dist as hdist

            def rank_all():
                return hdist.fullrank_topk_sharded(adj, out_u, out_i, users, ev["indptr"], ev["indices"], ev["n_items"], EVAL_K,
                                                   return_stats=True)
        else:
            user_tab, item_tab = out_u[:ev["n_own"]].contiguous(), out_i.contiguous()

            def rank_all():
                return E.fullrank_topk(user_tab, item_tab, users, ev["indptr"], ev["indices"], EVAL_K, mode="exact", engine="auto",
                                       return_stats=True)
        times, stats = [], None
        for it in range(iters + 1):
            job.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ids, sc, stats = rank_all()
            host_ids = ids.cpu()  # the [n_test, K] id matrix is what the reference's metric code consumes
            e1.record()
            torch.cuda.synchronize()
            if it > 0:
                times.append(e0.elapsed_time(e1))
        ms = sum(times) / len(times)
        n_users_total = ev["n_own"]
        if world > 1:
            t = torch.tensor([ms, float(ev["n_own"])], device=dev, dtype=torch.float64)
            tmax = t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            ms, n_users_total = float(tmax[0]), int(t[1])
        # Recall@20 / NDCG@20 of this rank's users through the reference's metric arithmetic (util/evaluation.py), users
        # with held-out items only, exactly like GraphRecommender.test iterates data.test_set; outside the timed region
        has = np.diff(ev["truth_indptr"]) > 0
        sel = np.nonzero(has)[0]
        ptr = np.zeros(sel.size + 1, dtype=np.int64)
        np.cumsum(np.diff(ev["truth_indptr"])[sel], out=ptr[1:])
        keep = np.repeat(has, np.diff(ev["truth_indptr"]))
        torch.cuda.synchronize()
        t_m = time.perf_counter()
        measures = E.ranking_evaluation_device(ptr, ev["truth_items"][keep], ids[torch.from_numpy(sel).to(dev)], [EVAL_K]) if sel.size else []
        torch.cuda.synchronize()
        measure_s = time.perf_counter() - t_m
        s = stats.tolist()
        flops = 2.0 * D * ev["n_items"] * n_users_total
        tf = flops / (ms * 1e-3) / 1e12
        return {"users_per_s": n_users_total / ms * 1e3, "ms": ms, "users": n_users_total, "items": ev["n_items"], "k": EVAL_K,
                "mode": "exact", "d2h_bytes": int(host_ids.numel() * 4), "score_tflops": tf,
                "roofline": eval_roofline(workload, world, n_users_total, ev["n_items"], ms),
                "candidates_per_user": s[0] / max(ev["n_own"], 1), "rescored_per_user": s[1] / max(ev["n_own"], 1),
                "fallback_users": s[2], "tensor_error_ppm_of_bound": s[3], "metrics_rank0": [m.strip() for m in measures], "metrics_users_rank0": int(sel.size),
                "metrics_s": measure_s}


def run_eval_facade(job, model, facade, iters=3):
    """The reference's evaluation call on the facade: ``GraphRecommender.test`` body (evaluation.test -> rec_list dict) and
    ``ranking_evaluation`` on ``data.test_set``, timed like ``base/graph_recommender.py:120-125`` times it."""
    import types

    import torch

    from hypergraph_diffusion_for_recommendation_b200 import evaluation as E

    with torch.no_grad():
        out_u, out_i = model()[:2]
        rec = types.SimpleNamespace(data=facade, max_N=EVAL_K)
        times = []
        for it in range(iters + 1):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev = E.EvalData(facade, device=job.dev) if getattr(rec, "_hgr_eval_data", None) is None else rec._hgr_eval_data
            rec._hgr_eval_data = ev
            ids, sc = E.fullrank_topk(out_u.contiguous(), out_i.contiguous(), ev.test_users, ev.train_indptr, ev.train_indices, EVAL_K,
                                      mode="refquirk")
            ids.cpu()
            torch.cuda.synchronize()
            if it > 0:
                times.append(time.perf_counter() - t0)
        ms = 1e3 * sum(times) / len(times)
        t_m = time.perf_counter()
        measures = E.ranking_evaluation_device(ev.truth_indptr, ev.truth_items, ids, [EVAL_K])
        measure_s = time.perf_counter() - t_m
        n = int(ev.test_users.numel())
        return {"users_per_s": n / ms * 1e3, "ms": ms, "users": n, "items": int(facade.n_items), "k": EVAL_K, "mode": "refquirk",
                "metrics": [m.strip() for m in measures], "metrics_s": measure_s,
                "roofline": eval_roofline("facade", 1, n, int(facade.n_items), ms)}


def summarise(line):
    """An extra_configs entry: the contract keys of one leg without the long notes."""
    keep = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "config",
            "e2e", "gpu_launches", "clocks", "cpu_baseline", "eval", "exchange", "graph_build", "loss")
    out = {k: line[k] for k in keep if k in line}
    r = line.get("roofline") or {}
    out["roofline"] = {k: r.get(k) for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "launch_ms", "launches_timed", "spmm_share_of_step")}
    out["roofline"]["l2_to_sm_gbs"] = (r.get("l2_to_sm") or {}).get("gbs")
    return out


def run_ours(args):
    import torch

    job = Job(args)
    line = measure(job, args.workload, args.model, args.steps, args.warmup, args.cpu_steps, not args.no_cpu_baseline, primary=True)
    if not args.no_extra and args.workload == "c5w":
        extras = []
        legs = EXTRA_LEGS if job.world == 1 else (("c4", "hgnn_hd3"),)
        for wl, mdl in legs:
            ex = measure(job, wl, mdl, min(args.steps, 10), max(3, min(args.warmup, 5)), 1, not args.no_cpu_baseline, primary=False)
            if ex is not None:
                extras.append(summarise(ex))
        parity = None
        if job.world > 1:
            from hypergraph_diffusion_for_recommendation_b200 import dist_check

            parity = dist_check.parity_check(job.rank, job.world, job.dev)
        if line is not None:
            line["extra_configs"] = extras
            if parity is not None and line.get("parity_at_scale"):
                parity["checks"].update({k: v for k, v in line["parity_at_scale"].items() if k != "multicast"})
                parity["ok"] = all(parity["checks"].values())
            line["parity"] = parity
    if line is not None:
        emit(line)
    torch.cuda.synchronize()
    job.close()


_JSON_FD = None


def _reserve_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner with printf when the
    first communicator comes up), so everything else is sent to stderr and the line goes out through a saved descriptor."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def main():
    args = parse_args()
    _reserve_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
