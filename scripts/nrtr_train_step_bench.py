#!/usr/bin/env python
"""NRTR recogniser training step (BASELINE config 3): img [128, 3, 32, 128] seeded N(0, 1), seeded random 5-12-character DICT90
labels, NRTR.forward_train (TFLoss), backward, Adam 1e-4 -- two arms timed alternately in one process with CUDA events, TF32 off:

  native   the encoder and the teacher-forced decoder on tpspp_attn_train_fwd/_bwd and tpspp_linear_fwd/_bwd (nrtr_train)
  library  the same step with the attention as torch ops (the reference's masked soft-max) and the dense layers as F.linear

The backbone (layers 3-5 and BatchNorm in training mode: torch ops) and TPS_PP (its native training path) are the same in both.
Also reported: both arms' loss on one batch at dropout 0 (same weights).  --profile adds a per-kernel device-time table of the
native step from torch.profiler, in a run of its own after the timing.  Writes --out (default profiles/r05_nrtr_train_step.json).
Multi-GPU: python -m torch.distributed.run --nproc-per-node N scripts/nrtr_train_step_bench.py (parallel.GradBucket all-reduce)."""
import argparse
import json
import os
import random
import subprocess
import sys
import types

import torch
import torch.distributed as dist
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tps_pp_b200 as T  # noqa: E402
from tps_pp_b200 import functional as TF, nrtr_train, parallel as PAR  # noqa: E402
from tps_pp_b200.recognizer import DICT90  # noqa: E402
from oracle import tpspp_oracle as O  # noqa: E402


def lib_attention(q, k, v, heads, len_q, len_k, temperature, kv_lens=None, causal=False, dropout_p=0.0):
    """``_attn_lib``'s masked soft-max (transformer_module.py:24-34) with the reference's attention dropout, on torch ops."""
    b = q.shape[0] // len_q
    if isinstance(kv_lens, TF.AttnLengths):
        kv_lens = kv_lens.host
    qq = q.reshape(b, len_q, heads, 64).transpose(1, 2)
    kk = k.reshape(b, len_k, heads, 64).transpose(1, 2)
    vv = v.reshape(b, len_k, heads, 64).transpose(1, 2)
    a = torch.matmul(qq / temperature, kk.transpose(2, 3))
    mask = torch.ones((b, 1, len_q, len_k), dtype=torch.bool, device=q.device)
    if kv_lens is not None:
        mask = mask & (torch.arange(len_k, device=q.device) < torch.tensor(list(kv_lens), device=q.device)[:, None])[:, None, None, :]
    if causal:
        mask = mask & torch.ones((len_q, len_k), dtype=torch.bool, device=q.device).tril()
    p = F.dropout(F.softmax(a.masked_fill(~mask, float("-inf")), dim=-1), dropout_p, training=dropout_p > 0)
    return torch.matmul(p, vv).transpose(1, 2).reshape(b * len_q, heads * 64)


LIBRARY_OPS = types.SimpleNamespace(linear=F.linear, attention=lib_attention, AttnLengths=TF.AttnLengths)


def gpu_info(dev):
    info = {"gpu": torch.cuda.get_device_name(dev)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(dev.index)],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = r.stdout.strip()
    except Exception as e:          # the figure is still reported; the card's limit is then unknown
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_nrtr_train_step.json"))
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(0)
    rec = T.build_recognizer(dict(
        type="NRTR",
        backbone=dict(type="ResNetABI_v2_large", arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]),
        tpsnet=dict(type="TPS_PP"), encoder=dict(type="NRTREncoder"), decoder=dict(type="NRTRDecoder"), loss=dict(type="TFLoss"),
        label_convertor=dict(type="AttnConvertor", dict_type="DICT90", with_unknown=True, max_seq_len=40)))
    rec.tpsnet.load_state_dict(O.trained_like_state(3), strict=True)
    rec = rec.to(dev).train()
    B = args.batch
    g = torch.Generator().manual_seed(1000 + rank)
    img = torch.randn((B, 3, 32, 128), generator=g).to(dev)
    rng = random.Random(1000 + rank)
    metas = [dict(text="".join(rng.choice(DICT90) for _ in range(rng.randint(5, 12))), valid_ratio=1.0) for _ in range(B)]
    bucket = PAR.GradBucket(rec.parameters())
    opt = torch.optim.Adam(rec.parameters(), lr=1e-4)

    def use(ops):
        nrtr_train.TF = ops

    def loss_of():
        return rec(img, metas, return_loss=True)["loss_ce"].mean()

    # both arms' loss on the same weights and batch at dropout 0 (the BatchNorm running statistics are restored after)
    buffers = {k: v.clone() for k, v in rec.named_buffers()}
    enc_p, dec_p = rec.encoder.dropout, rec.decoder.dropout.p
    rec.encoder.dropout, rec.decoder.dropout.p = 0.0, 0.0
    loss0, native_flag = {}, {}
    with torch.no_grad():
        for name, ops in (("native", TF), ("library", LIBRARY_OPS)):
            use(ops)
            loss0[name] = float(loss_of())
            native_flag[name] = rec.last_train_native
    rec.encoder.dropout, rec.decoder.dropout.p = enc_p, dec_p
    with torch.no_grad():
        for k, v in rec.named_buffers():
            v.copy_(buffers[k])

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = {"native": [], "library": []}
    for it in range(args.warmup + args.steps):
        for name, ops in (("native", TF), ("library", LIBRARY_OPS)):
            use(ops)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            ev[0].record()
            bucket.zero()
            loss_of().backward()
            bucket.all_reduce_mean()
            opt.step()
            ev[1].record()
            torch.cuda.synchronize()
            if it >= args.warmup:
                times[name].append(ev[0].elapsed_time(ev[1]))
    use(TF)
    kernels = None
    if args.profile and rank == 0:
        from torch.profiler import ProfilerActivity, profile
        nprof = 3
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(nprof):
                bucket.zero()
                loss_of().backward()
                opt.step()
            torch.cuda.synchronize()
        rows = sorted(((e.key, e.self_device_time_total / nprof, e.count // nprof) for e in prof.key_averages()), key=lambda r: -r[1])
        kernels = [dict(name=k[:160], us_per_step=round(us, 1), calls_per_step=n) for k, us, n in rows if us > 0]
    ms = {k: sum(v) / len(v) for k, v in times.items()}
    t = torch.tensor([ms["native"], ms["library"]], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        res = {"metric": "nrtr_train_step", "n_gpus": world, "batch_per_gpu": B, "steps": args.steps, "warmup": args.warmup,
               "native_ms_per_step": t[0].item(), "library_ms_per_step": t[1].item(),
               "native_img_per_s": world * B / (t[0].item() * 1e-3), "library_img_per_s": world * B / (t[1].item() * 1e-3),
               "native_step_ms_each": [round(x, 3) for x in times["native"]], "library_step_ms_each": [round(x, 3) for x in times["library"]],
               "loss_dropout0": loss0, "last_train_native": native_flag, "tf32": False, **gpu_info(dev)}
        if kernels is not None:
            res["kernels_native_step"] = kernels
            res["device_us_per_native_step"] = round(sum(k["us_per_step"] for k in kernels), 1)
        print(json.dumps({k: v for k, v in res.items() if k != "kernels_native_step"}))
        if kernels is not None:
            for k in kernels[:40]:
                print("%9.1f us %4d x  %s" % (k["us_per_step"], k["calls_per_step"], k["name"][:120]))
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
