"""The propagation kernel on ONE rank's block of the row-partitioned 10 M x 2 M x 1 B graph (BASELINE configs[4]), run on a
single GPU without any communication, so that it can be profiled with ncu (multi-rank commands cannot):

    python tools/shard_probe.py [--world 8] [--rank 0] [--iters 5]

The block is A[own rows, :] with 1.5 M rows, ~250 M nonzeros and 12 M columns; X is the gathered [12 M, 64] table (3 GB)."""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hypergraph_diffusion_for_recommendation_b200 import dist as hdist  # noqa: E402
from hypergraph_diffusion_for_recommendation_b200 import ops  # noqa: E402
from hypergraph_diffusion_for_recommendation_b200.graph import DeviceCSR  # noqa: E402
from hypergraph_diffusion_for_recommendation_b200.synth import powerlaw_interactions_device  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--world", type=int, default=8)
    ap.add_argument("--rank", type=int, default=0)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--schedules", default="binned,windowed,spread", help="work schedules to time (graph.work_schedule)")
    ap.add_argument("--splits", default="fixed", help="split plans: fixed | window[:shift[:min_seg]]")
    ap.add_argument("--chunks", default="0", help="chunk_nnz values of the split plan to time (0 = the default rule)")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    U, I, E = 1_250_000 * args.world, 250_000 * args.world, 125_000_000 * args.world
    t0 = time.time()
    u, i = powerlaw_interactions_device(U, I, E, dev, seed=1234)
    part = hdist.Partition(U, I, args.world)
    indptr, indices, values = hdist.local_block(part, args.rank, u, i)
    del u, i
    torch.cuda.empty_cache()
    block = DeviceCSR(indptr, indices, values, (part.n_loc, part.n_glob))
    torch.cuda.synchronize()
    print("block %d of %d: rows %d cols %d nnz %d, heavy rows %d, built in %.1f s" % (
        args.rank, args.world, part.n_loc, part.n_glob, block._nnz(), block.desc.n_heavy_rows, time.time() - t0), flush=True)
    x = torch.randn(part.n_glob, 64, device=dev)
    deg = (indptr[1:] - indptr[:-1])
    for name, dsel in (("user rows", deg[:part.up]), ("item rows", deg[part.up:])):
        tot = int(dsel.sum())
        line = ["%s: %d rows, %d nnz" % (name, dsel.numel(), tot)]
        for lo, hi in ((0, 64), (64, 256), (256, 1024), (1024, 4096), (4096, 16384), (16384, 1 << 40)):
            m = (dsel >= lo) & (dsel < hi)
            line.append("[%d,%s): %d rows %.1f%% nnz" % (lo, hi if hi < (1 << 40) else "inf", int(m.sum()), 100.0 * int(dsel[m].sum()) / max(tot, 1)))
        print("  " + " | ".join(line), flush=True)
    del block
    made = None
    for chunk, split, sched in ((int(c), sp, s) for c in args.chunks.split(",") for sp in args.splits.split(",")
                                for s in args.schedules.split(",")):
        if made != (chunk, split):
            block = None
            torch.cuda.empty_cache()
            t0 = time.time()
            block = DeviceCSR(indptr, indices, values, (part.n_loc, part.n_glob), chunk_nnz=chunk or None, split=split)
            torch.cuda.synchronize()
            made = (chunk, split)
            print("split %s chunk_nnz %d: heavy rows %d, chunks %d, plan %.2f s" % (block.split, block.chunk_nnz, block.desc.n_heavy_rows,
                                                                               block.desc.n_chunks, time.time() - t0), flush=True)
        block.set_schedule(sched)
        print("schedule %s" % sched, flush=True)
        for _ in range(2):
            y = ops.spmm_raw(block, x)
        ts = []
        for _ in range(args.iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            y = ops.spmm_raw(block, x)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ms = sorted(ts)[len(ts) // 2]
        nnz = block._nnz()
        alg = 8 * (part.n_loc + 1) + 8 * nnz + 256 * nnz + 256 * part.n_loc
        print("spmm median %.3f ms | %.1f Gnnz/s | algorithmic %.1f GB -> %.0f GB/s" % (ms, nnz / ms / 1e6, alg / 1e9, alg / ms / 1e6), flush=True)


if __name__ == "__main__":
    main()
