"""Quick device probe: SpMM time / algorithmic GB/s on synthetic shapes (not the bench contract)."""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hypergraph_diffusion_for_recommendation_b200 import ops  # noqa: E402
from hypergraph_diffusion_for_recommendation_b200.synth import norm_adj_from_pairs_torch, powerlaw_interactions_device  # noqa: E402


def algorithmic_bytes(n, nnz, d):
    gather = 4 * d * n if 4 * d * n <= 64e6 else 4 * d * nnz
    return 8 * (n + 1) + 8 * nnz + gather + 4 * d * n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="52000x92000x3000000,1250000x250000x125000000")
    ap.add_argument("--chunks", default="0")
    ap.add_argument("--schedules", default="binned,windowed")
    ap.add_argument("--splits", default="fixed", help="split plans to time: fixed | window[:shift[:min_seg]] (graph.DeviceCSR)")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--d", type=int, default=64)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for shape in args.shapes.split(","):
        U, I, E = (int(v) for v in shape.split("x"))
        t0 = time.time()
        u, i = powerlaw_interactions_device(U, I, E, dev)
        torch.cuda.synchronize()
        from hypergraph_diffusion_for_recommendation_b200.graph import DeviceCSR

        base = norm_adj_from_pairs_torch(u, i, U, I, chunk_nnz=1 << 30)
        n, nnz = U + I, base._nnz()
        x = torch.randn(n, args.d, device=dev)
        y_seq = ops.spmm_raw(base, x).clone()  # every row accumulated sequentially (no split plan)
        for chunk, split in ((int(c), sp) for c in args.chunks.split(",") for sp in args.splits.split(",")):
            torch.cuda.synchronize()
            t1 = time.time()
            adj = DeviceCSR(base.indptr, base.indices, base.values, base.shape, symmetric=True, chunk_nnz=chunk or None, split=split)
            torch.cuda.synchronize()
            t2 = time.time()
            deg = adj.indptr[1:] - adj.indptr[:-1]
            print("shape %s nnz %d plan %.2fs split %s chunk %d heavy_rows %d chunks %d maxdeg %d" % (
                shape, nnz, t2 - t1, adj.split, adj.chunk_nnz, adj.desc.n_heavy_rows, adj.desc.n_chunks, int(deg.max())), flush=True)
            adj.set_schedule("binned")
            y_ref = ops.spmm_raw(adj, x).clone()
            err = ((y_ref - y_seq).abs().amax(1) / y_seq.abs().amax(1).clamp(min=1e-30)).max()
            print("  vs sequential rows: worst row-wise relative difference %.2e" % float(err), flush=True)
            for sched in args.schedules.split(","):
                adj.set_schedule(sched)
                for _ in range(3):
                    y = ops.spmm_raw(adj, x)
                if not torch.equal(y, y_ref):
                    print("  %s: RESULT DIFFERS from the binned schedule (max abs %.3e)" % (sched, float((y - y_ref).abs().max())))
                times = []
                for _ in range(args.iters):
                    flush.fill_(1)
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record()
                    y = ops.spmm_raw(adj, x)
                    e.record()
                    torch.cuda.synchronize()
                    times.append(s.elapsed_time(e))
                ms = sorted(times)[len(times) // 2]
                b = algorithmic_bytes(n, nnz, args.d)
                print("  %-11s | spmm median %.3f ms min %.3f ms | alg %.1f MB -> %.0f GB/s | %.1f Gnnz/s" % (
                    sched, ms, min(times), b / 1e6, b / ms / 1e6, nnz / ms / 1e6), flush=True)
            del adj, y
        del base, x, y_seq


if __name__ == "__main__":
    main()
