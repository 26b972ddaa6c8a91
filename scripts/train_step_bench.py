#!/usr/bin/env python
"""Training-step timing of the rectifier (BASELINE config 3, rectifier part): forward + backward +
one flat-bucket NCCL all-reduce + Adam, batch 128 per GPU.  The loss is a synthetic regression on `output`; the whole
recogniser's step (NRTR.forward_train, TFLoss) is scripts/nrtr_train_step_bench.py.  Launch: python scripts/train_step_bench.py  or
python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/train_step_bench.py"""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tps_pp_b200 as T  # noqa: E402
from tps_pp_b200 import parallel as PAR  # noqa: E402
from bench import _trained_like_  # noqa: E402


def main():
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, steps, warm = 128, 10, 3
    convs = "library" if "--library-convs" in sys.argv else "native"
    m = T.TPS_PP().to(dev).train()
    m.train_convs = convs
    m.train_linears = "library" if ("--library-linears" in sys.argv or convs == "library") else "native"
    _trained_like_(m)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    bucket = PAR.GradBucket(m.parameters())
    opt = torch.optim.Adam(m.parameters(), lr=1e-4)      # schedule_adam_step_12e.py:1
    g = torch.Generator(device=dev).manual_seed(rank)
    x = torch.randn((B, 64, 16, 64), device=dev, generator=g)
    o0 = torch.randn((B, 32, 32, 128), device=dev, generator=g)
    o1 = torch.randn((B, 32, 32, 128), device=dev, generator=g)
    tgt = torch.randn((B, 64, 16, 64), device=dev, generator=g)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    t_total = t_ar = t_fwd = 0.0
    for it in range(warm + steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev[0].record()
        bucket.zero()
        r = m(x, [o0, o1])
        loss = (r["output"] - tgt).square().mean()
        ev[4].record()
        loss.backward()
        ev[1].record()
        bucket.all_reduce_mean()
        ev[2].record()
        opt.step()
        ev[3].record()
        torch.cuda.synchronize()
        if it >= warm:
            t_total += ev[0].elapsed_time(ev[3]); t_ar += ev[1].elapsed_time(ev[2]); t_fwd += ev[0].elapsed_time(ev[4])
    # the same step with forward + backward captured in ONE CUDA graph (the eager loop above is bound by ~2 ms of Python /
    # autograd / ctypes launch overhead per step): zero the bucket, forward, loss, backward are replayed; the all-reduce and the
    # optimiser step stay outside the graph
    graph_ms = None
    loss_value = float(loss.detach())
    del r, loss                                  # the eager autograd graph (its AccumulateGrad nodes live on the default stream) must be gone
    if "--no-graph" not in sys.argv:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):            # warm the capture stream's allocator / lazy initialisations
            bucket.zero()
            for _ in range(2):
                (m(x, [o0, o1])["output"] - tgt).square().mean().backward()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            bucket.flat.zero_()
            r = m(x, [o0, o1])
            loss = (r["output"] - tgt).square().mean()
            loss.backward()
        del r, loss
        t_g = 0.0
        for it in range(warm + steps):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev[0].record()
            graph.replay()
            bucket.all_reduce_mean()
            opt.step()
            ev[3].record()
            torch.cuda.synchronize()
            if it >= warm:
                t_g += ev[0].elapsed_time(ev[3])
        graph_ms = t_g / steps
    if "--profile" in sys.argv and rank == 0:
        # per-kernel device time of one training step (CUPTI, not ncu: warm caches, real overlap) -> stdout table
        from torch.profiler import profile, ProfilerActivity
        nprof = 4
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(nprof):
                bucket.zero()
                r = m(x, [o0, o1])
                loss = (r["output"] - tgt).square().mean()
                loss.backward()
                opt.step()
            torch.cuda.synchronize()
        rows = sorted(((e.key, e.self_device_time_total / nprof, e.count // nprof) for e in prof.key_averages()),
                      key=lambda r: -r[1])
        tot = sum(r[1] for r in rows)
        print("# per-step device time %.1f us over %d kernel names" % (tot, len(rows)))
        for k, us, n in rows[:70]:
            print("%9.1f us %4d x  %s" % (us, n, k[:150]))
    t = torch.tensor([t_total / steps, t_ar / steps, t_fwd / steps, graph_ms if graph_ms is not None else 0.0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        best = t[3].item() if graph_ms is not None else t[0].item()
        print(json.dumps({"metric": "tps_pp_train_step", "n_gpus": world, "batch_per_gpu": B, "ms_per_step": best,
                          "cuda_graph": graph_ms is not None, "eager_ms_per_step": t[0].item(),
                          "allreduce_ms": t[1].item(), "eager_forward_ms": t[2].item(), "img_per_s": world * B / (best * 1e-3),
                          "grad_bucket_bytes": bucket.flat.numel() * 4, "loss": loss_value, "training_stages": m.training_stages,
                          "head": f"14 ConvModules: {convs} forward+backward (fp32-level); 16 dense layers (CBAM/DGAB/localisation/score): "
                                  f"{m.train_linears} forward+backward; LayerNorm/softmax/GELU/elementwise: torch ops; warp fwd/bwd native"}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
