#!/usr/bin/env python
"""Headline benchmark: TPS_PP rectifier forward (BASELINE.json configs[1]) -- img/s and the fused
warp kernel's HBM roofline fraction.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step = one ``TPS_PP.forward`` over a batch of 256 synthetic feature maps per GPU
(x [256,64,16,64], outs 2x[256,32,32,128], fp32, F=32 -- the only geometry the reference module
accepts, SURVEY F4).  One process per GPU, the batch is sharded with no collective on the data
path (weak scaling); timing is CUDA events, max over ranks.  See DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH_PER_GPU = 256
WORKLOAD = "TPS_PP rectifier alone fp32 forward, batch 256/GPU, F=32 (2x16) control points, x[64,16,64]+outs 2x[32,32,128]"
# SURVEY 8(d): algorithmic bytes of the fused warp per image (TPS++ fp32, output + mp_img)
WARP_BYTES_PER_IMG = 1048576 + 262144 + 131072 + 256 + 262144 + 262144
TF32X3_CEILING = 1125.0 / 3.0      # TFLOP/s: nominal dense tf32 rate, three MMAs per fp32 product
STAGE_GFLOP_PER_IMG = 0.607        # stem 7.1 M + layer1 251.7 M + layer2 348.2 M (resnet_v2_large.py:109-135; 2 FLOP per MAC)
HEAD_GFLOP_PER_IMG = 0.82          # SURVEY 8(d): convs 720.6 M + DGAB/MLP 76.4 M + score 21.4 M + localization 1.1 M
WARP_CONST_BYTES = 131072 + 4900 + 8192
DUMP_LIMIT_BYTES = 60 * 10 ** 6        # array data of --dump-outputs: with the .npy headers the files stay under 64 MB


def _dump_outputs(path, arrays):
    """Write what a caller of the timed path received in its last step to path/<name>.npy as float32.  The arrays share
    their leading (batch) dimension; when together they exceed DUMP_LIMIT_BYTES, the same fixed, seeded sample of batch
    indices is kept from each, so two builds run with the same arguments write the same elements."""
    batch = next(iter(arrays.values())).shape[0]
    per_item = sum(t[0].numel() * 4 for t in arrays.values())
    keep = min(batch, DUMP_LIMIT_BYTES // per_item)
    idx = torch.from_numpy(np.sort(np.random.RandomState(0).choice(batch, keep, replace=False)))
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t[idx.to(t.device)].float().cpu().numpy())
    print(f"bench: wrote {', '.join(sorted(arrays))} of {keep} of {batch} items to {path}", file=sys.stderr, flush=True)


def _warp_traffic():
    """dram__bytes_read+write of one warp launch from the committed ncu capture (bench never runs under ncu)."""
    path = os.path.join(ROOT, "profiles", "warp_traffic.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
        return int(d["dram_bytes_per_launch"]) if int(d.get("batch", 0)) == BATCH_PER_GPU else None
    except Exception:
        return None


def _tensor_peak():
    """Dense bf16 TFLOP/s measured on this pool (sustained figure: the head runs inside a long step)."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            d = json.load(fh)
        return float(d.get("bf16_tflops_sustained") or d["bf16_tflops"]), "measured bf16 sustained (MEASURED_PEAKS.json)"
    except Exception:
        return 2250.0, "nominal dense bf16 (B200_PROFILING.md fallback)"


_MID = ["enc0", "enc1", "enc2", "enc3", "cbam", "dec0", "dec1", "dec2", "dec3", "localization+p_linear", "dgab_gate", "mlp_fused"]
_DOWN = (["down_fused(down0+down1+down2+down_feat)", "down0_1", "down1_1"],
         ["down0", "down1", "down2", "down0_1", "down1_1", "down_feat"])
_SCORE = (["score_fused(feat_linear.0+.1+qkt)"], ["feat_linear.0", "feat_linear.1", "score_qkt"])


def _launch_names(n):
    """Names of the library's launches of one forward, in order (the weight re-layout launch is skipped when the
    cached images are valid; the bf16 / fp32 modes and the A/B flags run the fused stages as separate launches)."""
    for down in _DOWN:
        for score in _SCORE:
            names = down + _MID + score + ["fused_warp"]
            if n == len(names):
                return names
            if n == len(names) + 1:
                return ["wprep"] + names
    return None


def _split_ceiling(head):
    """Tensor ceiling of the fp32-parity operand modes, TFLOP/s of algorithmic work: a product costs three tf32 MMAs in the
    all-tf32 3xTF32 form (nominal dense tf32 1125 / 3 = 375) and one tf32 + two bf16 MMAs -- two tf32-equivalents -- in the
    default mixed form (1125 / 2 = 562)."""
    return {"tc": (562.5, "tf32 main term + two bf16 correction MMAs = 2 tf32-equivalents per product: nominal dense tf32 1125 / 2"),
            "tc3x": (TF32X3_CEILING, "three tf32 MMAs per product: nominal dense tf32 1125 / 3")}.get(head, (None, None))


def _dominant(launch_ms, batch, tpeak, tpeak_src, step_ms, head):
    names = _launch_names(len(launch_ms)) if launch_ms else None
    if names is None:
        return None
    i = max(range(len(launch_ms)), key=lambda k: launch_ms[k])
    out = {"kernel": names[i], "avg_launch_ms": launch_ms[i], "share_of_step": launch_ms[i] / step_ms,
           "per_launch_ms": dict(zip(names, [round(v, 4) for v in launch_ms]))}
    ceil, ceil_what = _split_ceiling(head)

    def enc0_entry(ms):
        gflop = 2 * 1024 * 1728 * 64 * batch / 1e9
        ach = gflop / ms                                 # GFLOP / ms = TFLOP/s
        return {"what": "conv_tma_kernel<3>: 3x3 conv 192->64 at 16x64 (enc0)", "bound": "tensor", "avg_launch_ms": ms, "achieved": ach,
                "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak, "peak_source": tpeak_src, "gflop_per_launch": gflop,
                "frac_of_split_fp32_ceiling": ach / ceil if ceil else None, "split_fp32_ceiling": ceil, "split_fp32_ceiling_is": ceil_what}
    if names[i] == "enc0":
        out.update(enc0_entry(launch_ms[i]))
    elif names[i].startswith("down_fused"):
        # o0 + o1 + x read once, f0 / f1 / f2 / feat_grid written once (DESIGN.md section 4): 4,718,592 B per image
        nbytes = batch * 4 * (2 * 32 * 4096 + 64 * 1024 + 2 * 64 * 4096 + 64 * 1024 + 64 * 4096)
        peak, peak_src = _peaks()
        ach = nbytes / (launch_ms[i] * 1e-3) / 1e9
        out.update({"what": "down_fused_kernel: down0 + down1 + down2 + down_feat in one pass (four 1x1 convolutions, TMEM-chained)",
                    "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
                    "bytes_per_launch": nbytes})
    if "enc0" in names and names[i] != "enc0":
        out["largest_tensor_bound_kernel"] = enc0_entry(launch_ms[names.index("enc0")])
    return out


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle-reason samples taken DURING the timed region.

    In-process NVML (nvidia_ml_py) polled every 2 ms from a thread: a timed region of 20 steps lasts ~40 ms, which a
    freshly spawned ``nvidia-smi -lms`` (first line after >100 ms, longer with 8 ranks starting one each) misses."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.index = index
        self.sm, self.bits, self.mx = [], 0, None
        self._stop = threading.Event()
        self.t = None
        self.h = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _sample(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            self.bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))

    def _run(self):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception:
                return
            time.sleep(0.002)

    def start(self):
        if self.h is None:
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml unavailable"]}
        self._stop.set()
        self.t.join(timeout=1.0)
        reasons = sorted(nm for bit, nm in self.REASONS.items() if self.bits & bit)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx,
                "samples": len(self.sm), "reasons": reasons}


def _dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def _bind_to_gpu_cpus(local: int):
    """Pin this rank (and, by first touch, its pinned host buffers) to the CPUs NVML reports as local to its GPU: with
    several ranks per node the end-to-end path is bound by host memory / PCIe root traffic, and buffers that land on the
    other socket cross the inter-socket link on every copy.  Returns a short description for the JSON line."""
    if os.environ.get("TPSPP_BENCH_AFFINITY", "1") == "0" or not hasattr(os, "sched_setaffinity"):
        return "off"
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = None
        if torch.cuda.is_available():
            uuid = str(torch.cuda.get_device_properties(local).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode()) if uuid else pynvml.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [i for i in range(ncpu) if (int(words[i // 64]) >> (i % 64)) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return "none"
        os.sched_setaffinity(0, allowed)
        return f"{len(allowed)} cpus local to the GPU ({allowed[0]}-{allowed[-1]})"
    except Exception as e:  # noqa: BLE001 -- affinity is an optimisation, never a failure
        return f"unavailable ({type(e).__name__})"


def _cpu_reference(steps: int, warmup: int, batch: int):
    """The reference's CPU path (oracle port: same torch CPU ops the reference module calls,
    oracle/tpspp_oracle.py) on all host cores."""
    from oracle import tpspp_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = O.trained_like_state(3)
    x, o0, o1 = O.synthetic_tpspp_inputs(batch, seed=0)
    xs = (torch.from_numpy(x), [torch.from_numpy(o0), torch.from_numpy(o1)])
    consts = O.tpspp_constants()
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.tps_pp_forward(sd, xs[0], xs[1], dtype=torch.float32, sampler="torch", consts=consts)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    med = statistics.median(times)
    return batch / med, med * 1e3, cores


def _cpu_reference_image(steps: int, batch: int):
    """The reference's CPU path from the IMAGE: stem + layer1 + layer2 (oracle.backbone_stage_forward) then the rectifier --
    the CPU counterpart of our `from_image` / image-boundary `e2e` figures (bounded sample)."""
    from oracle import tpspp_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd_b, sd_t = O.trained_like_backbone_state(5), O.trained_like_state(3)
    img = O.synthetic_images(batch)
    consts = O.tpspp_constants()
    times = []
    with torch.no_grad():
        for i in range(1 + steps):
            t0 = time.perf_counter()
            xx, outs = O.backbone_stage_forward(sd_b, img, torch.float32)
            O.tps_pp_forward(sd_t, xx, outs, dtype=torch.float32, sampler="torch", consts=consts)
            dt = time.perf_counter() - t0
            if i >= 1:
                times.append(dt)
    med = statistics.median(times)
    return {"value": batch / med, "unit": "img/s", "cores": cores, "kind": "port",
            "sample": f"{steps} steps of batch {batch} (median {med * 1e3:.0f} ms): oracle stem + layer1 + layer2 + rectifier, torch CPU fp32"}


def run_reference(args):
    rank, world, _ = _dist_env()
    if rank != 0:
        return
    # same config as our arm: batch 256 per step, exactly --steps timed steps after --warmup untimed ones
    # (~0.65 s per step on the 16 host cores of the GPU box: the default 20 + 5 run takes ~20 s)
    steps = max(1, args.steps)
    warm = max(0, args.warmup)
    batch = args.batch if args.global_batch <= 0 else min(256, args.global_batch)     # bounded sample of the global batch
    ips, ms, cores = _cpu_reference(steps, warm, batch)
    line = {
        "impl": "reference", "metric": "tps_pp_rectified_img_per_s", "value": ips, "unit": "img/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong" if args.global_batch > 0 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": (WORKLOAD if batch == BATCH_PER_GPU and args.global_batch <= 0 else
                                WORKLOAD.replace("batch 256/GPU", f"global batch {args.global_batch} split over {args.gpus} GPU(s) (BASELINE configs[4] shard)"
                                                 if args.global_batch > 0 else f"batch {batch}/GPU (non-default shard size)")),
                   "global_batch": args.global_batch if args.global_batch > 0 else batch,
                   "sample": f"batch {batch} per step on host CPU, {cores} threads"},
        "cpu_baseline": {"value": ips, "unit": "img/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} steps of batch {batch} (median), torch CPU fp32, {cores} threads"},
        "e2e": {"value": ips, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        # CPU counterpart of our arm's image-boundary figures (its `e2e` and `from_image` start from the image and carry the
        # backbone stage's 0.6 GFLOP/img on top of the rectifier); `e2e` above stays the rectifier alone, as the contract says
        "from_image": _cpu_reference_image(3, min(batch, 128)),
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch.distributed as dist
    import tps_pp_b200 as T
    from tps_pp_b200 import _native as N

    rank, world, local = _dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the TPS++ hot path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # only with several ranks per node (at N = 1 the end-to-end path is not host-bound, and the CPU-baseline leg of this
    # process must keep every core)
    host_affinity = _bind_to_gpu_cpus(local) if world > 1 else "off (single rank)"
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N.device_info()     # fails loudly on a non-sm_100 device / missing library
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    B = args.batch
    strong = args.global_batch > 0
    if strong:      # BASELINE configs[4]: a fixed global batch split over the ranks (images are independent: no exchange)
        from tps_pp_b200.parallel import shard_bounds
        lo, hi = shard_bounds(args.global_batch, rank, world)
        B = hi - lo
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.randn((B, 64, 16, 64), device=dev, generator=gen)
    o0 = torch.randn((B, 32, 32, 128), device=dev, generator=gen)
    o1 = torch.randn((B, 32, 32, 128), device=dev, generator=gen)
    # "trained-like" weights (SURVEY F8): same deterministic numpy recipe as the parity tests, restated
    # here without importing the oracle into the measured path
    m = T.TPS_PP().to(dev).eval()
    _trained_like_(m)
    if args.head == "library":
        m.head_impl = "library"
    else:
        m.head_precision = {"tc": N.HEAD_TC, "tc3x": N.HEAD_TC, "fp32": N.HEAD_FP32, "bf16": N.HEAD_BF16}[args.head]
        if args.head == "tc3x":          # A/B: 3x3 convolutions as all-tf32 3xTF32 instead of tf32 + bf16 corrections
            m.head_flags |= N.HEAD_FLAG_TF32X3_CONV

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches = 0
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            m(x, [o0, o1])
        barrier()
        m.warp_events = []
        sampler = ClockSampler(local)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            r = m(x, [o0, o1])
            launches += N.last_launch_count() + m._last_head_launches
        e1.record()
        barrier()
        clocks = sampler.stop()
        total_ms = e0.elapsed_time(e1)
        warp_ms = [a.elapsed_time(b) for a, b in m.warp_events]
        m.warp_events = None
        if args.dump_outputs and rank == 0:
            _dump_outputs(args.dump_outputs, {k: v for k, v in r.items() if v is not None})
        del r

        # per-launch times of the head (CUDA events recorded by the library around each of its kernels), taken in a
        # separate short pass after the timed region so the event records cannot perturb `value`
        launch_ms = None
        if args.head != "library":
            import ctypes
            lib = N.lib()
            buf = (ctypes.c_float * 64)()
            cnt = ctypes.c_int(0)
            acc = None
            lib.tpspp_launch_profile(1)
            for _ in range(5):
                m(x, [o0, o1])
                if lib.tpspp_launch_profile_read(buf, 64, ctypes.byref(cnt)) == 0 and cnt.value > 0:
                    cur = [float(buf[i]) for i in range(cnt.value)]
                    acc = cur if acc is None or len(acc) != len(cur) else [p + q for p, q in zip(acc, cur)]
            lib.tpspp_launch_profile(0)
            if acc is not None:
                launch_ms = [v / 5.0 for v in acc]

        # ---- end-to-end through the public API with HOST buffers (pinned); every step's H2D copy of its
        # inputs and D2H read of its result are inside the timed region.  Copies run on their own streams
        # with two device buffer sets, so step i+1's upload overlaps step i's kernels (PCIe is the bound).
        def e2e_measure(dev_inputs, fn):
            """img/s-style timing of fn(*device inputs) -> result tensor with pinned HOST inputs and a HOST result: uploads on
            their own stream into two device buffer sets (step i+1's upload overlaps step i's kernels), download on a third."""
            hin = [t.cpu().pin_memory() for t in dev_inputs]
            dbuf = [tuple(torch.empty_like(t) for t in dev_inputs) for _ in range(2)]
            houts = [None, None]
            s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
            main = torch.cuda.current_stream(dev)
            ev_in = [torch.cuda.Event() for _ in range(2)]
            ev_free = [torch.cuda.Event() for _ in range(2)]
            ev_done = [torch.cuda.Event() for _ in range(2)]
            ev_read = [torch.cuda.Event() for _ in range(2)]

            def upload(i):
                k = i & 1
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_free[k])          # kernels of step i-2 no longer read this buffer set
                    for d, h in zip(dbuf[k], hin):
                        d.copy_(h, non_blocking=True)
                    ev_in[k].record(s_in)

            def run(nsteps):
                for k in range(2):
                    ev_free[k].record(main); ev_read[k].record(s_out)
                upload(0)
                for i in range(nsteps):
                    k = i & 1
                    if i + 1 < nsteps:
                        upload(i + 1)
                    main.wait_event(ev_in[k])
                    out = fn(*dbuf[k])
                    ev_done[k].record(main); ev_free[k].record(main)
                    if houts[k] is None:
                        houts[k] = torch.empty(out.shape, dtype=out.dtype).pin_memory()
                    with torch.cuda.stream(s_out):
                        s_out.wait_event(ev_done[k])
                        houts[k].copy_(out, non_blocking=True)
                        ev_read[k].record(s_out)
                    out.record_stream(s_out)
                main.wait_stream(s_out)

            run(3)
            nsteps = max(4, min(args.steps, 12))
            reps = []
            for _ in range(3):       # median of three timed repetitions: one 12-step window (~35 ms) is at the mercy of a single host hiccup
                barrier()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record()
                run(nsteps)
                f1.record()
                barrier()
                reps.append(f0.elapsed_time(f1))
            return statistics.median(reps), nsteps, sum(h.numel() * h.element_size() for h in hin), houts[0].numel() * houts[0].element_size()

        # (1) at the rectifier's own call boundary: three fp32 feature maps per image cross PCIe (1.31 MB/img)
        e2e_ms, e2e_steps, feat_h2d, feat_d2h = e2e_measure((x, o0, o1), lambda a, b, c: m(a, [b, c])["output"])

        # (2) at the image boundary (SURVEY 8f rank 3): img -> native stem + layer1 + layer2 (tpspp_stage_fwd) -> rectifier.
        # 49 KB per image go up instead of 1.31 MB; the step does MORE work (0.6 GFLOP/img of backbone convolutions).
        image = None
        if args.head in ("tc", "tc3x", "bf16"):
            bb = T.ResNetABI_v2_large(arch_settings=[3, 4, 6, 6, 3], strides=[1, 2, 2, 1, 2]).to(dev).eval()
            _trained_like_backbone_(bb)
            img = torch.randn((B, 3, 32, 128), device=dev, generator=gen)

            def from_image(im):
                xx, outs = bb.stage(im)
                return m(xx, outs)["output"]
            for _ in range(3):
                from_image(img)
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(args.steps):
                from_image(img)
            g1.record()
            barrier()
            img_ms = g0.elapsed_time(g1)
            stage_launch_ms = None
            import ctypes
            lib = N.lib()
            buf = (ctypes.c_float * 64)()
            cnt = ctypes.c_int(0)
            lib.tpspp_launch_profile(1)
            acc = None
            for _ in range(5):
                bb.stage(img)
                if lib.tpspp_launch_profile_read(buf, 64, ctypes.byref(cnt)) == 0 and cnt.value > 0:
                    cur = [float(buf[i]) for i in range(cnt.value)]
                    acc = cur if acc is None or len(acc) != len(cur) else [p + q for p, q in zip(acc, cur)]
            lib.tpspp_launch_profile(0)
            if acc is not None:
                stage_launch_ms = [round(v / 5.0, 4) for v in acc]
            ie_ms, ie_steps, ie_h2d, ie_d2h = e2e_measure((img,), from_image)
            image = {"img_ms": img_ms, "e2e_ms": ie_ms, "e2e_steps": ie_steps, "h2d": ie_h2d, "d2h": ie_d2h,
                     "stage_launch_ms": stage_launch_ms, "stage_native": bool(bb._last_stage_native)}

    with torch.no_grad():
        native_stages = dict(m.native_stages)
    t = torch.tensor([total_ms, e2e_ms, statistics.mean(warp_ms), image["img_ms"] if image else 0.0, image["e2e_ms"] if image else 0.0],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, warp_mean_ms, img_ms, img_e2e_ms = (float(v) for v in t.tolist())
    gB = args.global_batch if strong else world * B          # images all ranks process per step
    value = gB * args.steps / (total_ms * 1e-3)
    e2e_value = gB * e2e_steps / (e2e_ms * 1e-3)
    peak, peak_src = _peaks()
    # bf16 mode: feat_grid reaches the warp as bf16 planes (TPSPP_SRC0_BF16): 512 KB less per image
    warp_bytes = B * (WARP_BYTES_PER_IMG - (524288 if args.head == "bf16" else 0)) + WARP_CONST_BYTES
    achieved = warp_bytes / (warp_mean_ms * 1e-3) / 1e9
    tpeak, tpeak_src = _tensor_peak()
    head_ms = total_ms / args.steps - warp_mean_ms            # GFLOP / ms == TFLOP/s

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sb = min(B, 256)
        ips, ms, cores = _cpu_reference(steps=8, warmup=1, batch=sb)
        cpu = {"value": ips, "unit": "img/s", "cores": cores, "kind": "port",
               "sample": f"8 steps of batch {sb} (median {ms:.0f} ms), oracle torch-CPU fp32, {cores} threads"}
        if image:
            cpu["from_image"] = _cpu_reference_image(3, min(sb, 128))
    if rank == 0:
        feature_e2e = {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": feat_h2d, "d2h_bytes_per_step": feat_d2h, "reps": "median of 3 timed windows",
                       "steps": e2e_steps,
                       "boundary": "TPS_PP.forward(batch_img, outs): three fp32 feature maps per image cross PCIe (1.31 MB/img)"}
        if image:
            # headline e2e = the hot path from the HOST image: ResNetABI_v2_large.stage(img) (native stem + layer1 + layer2)
            # -> TPS_PP.forward -> host `output`; it carries 0.6 GFLOP/img more work than `value` (the rectifier alone)
            e2e_obj = {"value": gB * image["e2e_steps"] / (img_e2e_ms * 1e-3), "unit": "img/s",
                       "h2d_bytes_per_step": image["h2d"], "d2h_bytes_per_step": image["d2h"], "steps": image["e2e_steps"],
                       "reps": "median of 3 timed windows",
                       "boundary": "image: ResNetABI_v2_large.stage(img[B,3,32,128]) -> TPS_PP.forward(x, outs) -> output on the host "
                                   "(backbone stage in front of the call native, SURVEY 8f rank 3; 49 KB/img up, 256 KB/img down)"}
            image_obj = {"value": gB * args.steps / (img_ms * 1e-3), "unit": "img/s", "ms_per_step": img_ms / args.steps,
                         "what": "device-resident images -> stage -> rectifier (same timing rules as `value`)",
                         "stage_ms_per_step": img_ms / args.steps - total_ms / args.steps,
                         "stage_per_launch_ms": image["stage_launch_ms"], "stage_native": image["stage_native"],
                         "stage_gflop_per_img": STAGE_GFLOP_PER_IMG}
        else:
            e2e_obj, image_obj = feature_e2e, None
        # SURVEY 8f rank 2 / BASELINE configs[4] "+ NRTR inference": the recogniser's greedy decode behind the rectifier, as the
        # native incremental decode (tps_pp_b200.NRTRDecoder.forward_test) and as the reference's full-prefix recompute on
        # torch / cuBLAS fp32 ops -- same module, same random-init weights, same batch as the headline line; outside the timed region
        nrtr_obj = None
        if world == 1 and args.head == "tc" and not args.no_cpu_baseline:
            try:
                torch.manual_seed(0)
                dec = T.NRTRDecoder().to(dev).eval()
                enc = torch.randn((B, 64, 512), device=dev)         # 4 x 16 feature map of a 32 x 128 image after layer5

                def _time(fn, n_it):
                    fn(); fn()
                    torch.cuda.synchronize()
                    q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    q0.record()
                    for _ in range(n_it):
                        out_ = fn()
                    q1.record()
                    torch.cuda.synchronize()
                    return q0.elapsed_time(q1) / n_it, out_
                with torch.no_grad():
                    nat_ms, p_nat = _time(lambda: dec.forward_test(None, enc, None), 5)
                    lib_ms, p_lib = _time(lambda: dec.forward_test_library(None, enc, None), 1)
                nrtr_obj = {"what": "NRTRDecoder greedy decode, 6 layers x 512 x 8 heads, 40 steps, 64 source tokens, batch %d" % B,
                            "native_ms": nat_ms, "native_img_per_s": B / (nat_ms * 1e-3),
                            "reference_algorithm_on_cublas_fp32_ms": lib_ms, "speedup": lib_ms / nat_ms,
                            "argmax_agreement": float((p_nat.argmax(-1) == p_lib.argmax(-1)).float().mean()),
                            "native_path": "KV-cache incremental decode: tpspp_linear_ln_fwd (tcgen05 3xTF32, split-K, residual / GELU / next LayerNorm in the epilogue) + tpspp_attn_decode, one CUDA graph"}
                del dec, enc, p_nat, p_lib
            except Exception as e:  # noqa: BLE001 -- a secondary figure must not take the headline line down
                nrtr_obj = {"error": f"{type(e).__name__}: {e}"}
        line = {
            "metric": "tps_pp_rectified_img_per_s", "value": value, "unit": "img/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": ("bf16 operands + bf16 storage of the large intermediates (incl. feat_grid) in the ten 3x3 convolutions and the warp's "
                      "first source / f32 (3xTF32) elsewhere"
                      if args.head == "bf16" else "f32"),
            "data": "synthetic",
            "config": {"workload": (WORKLOAD if B == BATCH_PER_GPU and not strong else
                                    WORKLOAD.replace("batch 256/GPU", f"global batch {gB} split over {world} GPU(s) (BASELINE configs[4] shard)"
                                                     if strong else f"batch {B}/GPU (non-default shard size)")),
                       "global_batch": gB, "parallelism": f"batch-shard x{world}, no collective",
                       "l2": "inputs 302 MB/step > 126 MB L2 (no flush needed)",
                       "native_stages": native_stages, "weights": "trained-like synthetic (seed 3)", "head": args.head},
            "roofline": {"kernel": "warp_fwd_staged_kernel<dual>", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": _warp_traffic() if (B == BATCH_PER_GPU and args.head != "bf16") else None, "peak_source": peak_src,
                         "bytes_per_launch": warp_bytes, "avg_launch_ms": warp_mean_ms,
                         "warp_only_img_per_s": B / (warp_mean_ms * 1e-3)},
            # everything before the warp (convs, DGAB, localization, score): SURVEY 8(d) counts 0.82 GFLOP/img of
            # dense contractions.  The fp32-parity modes spend several MMAs per product (split operands, _split_ceiling):
            # the fraction of the measured bf16 peak and the fraction of the mode's own ceiling are both reported.
            "roofline_head": {"kernels": "conv_tma_kernel / conv_ts_kernel / lin_tma_kernel / conv_tc_kernel / dgab_warp_kernel / loc_p1_kernel / cbam_kernel",
                              "bound": "tensor", "achieved": HEAD_GFLOP_PER_IMG * B / head_ms, "peak": tpeak,
                              "unit": "TFLOP/s", "frac": HEAD_GFLOP_PER_IMG * B / head_ms / tpeak,
                              "frac_of_split_fp32_ceiling": (HEAD_GFLOP_PER_IMG * B / head_ms / _split_ceiling(args.head)[0]
                                                             if _split_ceiling(args.head)[0] else None),
                              "split_fp32_ceiling": _split_ceiling(args.head)[0], "split_fp32_ceiling_is": _split_ceiling(args.head)[1],
                              "peak_source": tpeak_src, "gflop_per_img": HEAD_GFLOP_PER_IMG,
                              "avg_head_ms": head_ms, "share_of_step": head_ms / (total_ms / args.steps)},
            # the single largest kernel of the step, timed live (see above): enc0 = 3x3 conv 192 -> 64 at 16x64,
            # 2 * 1024 * 1728 * 64 FLOP per image, three TF32 MMAs per product in the default mode
            "roofline_dominant": _dominant(launch_ms, B, tpeak, tpeak_src, total_ms / args.steps, args.head),
            "cpu_baseline": cpu,
            "e2e": e2e_obj,
            "e2e_feature_boundary": feature_e2e,
            "from_image": image_obj,
            "nrtr_decode": nrtr_obj,
            "gpu_launches": launches, "clocks": clocks, "host_affinity": host_affinity,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _trained_like_backbone_(bb):
    """Deterministic stage weights (numpy legacy RNG, seed 5): He-uniform convolutions, BatchNorm with non-trivial affine
    parameters and running statistics (residual branch damped) -- the recipe of the parity tests
    (oracle.trained_like_backbone_state), restated so the measured path does not import the oracle."""
    import math
    rs = np.random.RandomState(5)
    new = {}
    for k, v in bb.state_dict().items():
        if k.split(".")[0] not in ("conv1", "bn1", "layer1", "layer2"):
            continue
        shape = tuple(v.shape)
        if k.endswith("num_batches_tracked"):
            new[k] = torch.tensor(100, dtype=torch.int64)
        elif k.endswith("running_var"):
            new[k] = torch.from_numpy(rs.uniform(0.5, 1.5, shape).astype(np.float32))
        elif k.endswith("running_mean"):
            new[k] = torch.from_numpy((0.1 * rs.standard_normal(shape)).astype(np.float32))
        elif len(shape) == 4:
            bound = math.sqrt(6.0 / int(np.prod(shape[1:])))
            new[k] = torch.from_numpy(rs.uniform(-bound, bound, shape).astype(np.float32))
        elif k.endswith(".weight"):
            lo, hi = (0.1, 0.3) if ".bn2." in k else (0.6, 1.4)
            new[k] = torch.from_numpy(rs.uniform(lo, hi, shape).astype(np.float32))
        else:
            new[k] = torch.from_numpy((0.1 * rs.standard_normal(shape)).astype(np.float32))
    bb.load_state_dict(new, strict=False)


def _trained_like_(m):
    """Deterministic synthetic 'trained-like' weights (He/Xavier-uniform from numpy's legacy RNG, live
    localisation ReLU, tiny fc2 weight, smooth non-affine bias field) -- see DESIGN.md 'Synthetic weights'."""
    import math
    rs = np.random.RandomState(3)
    sd = m.state_dict()
    relu_fed = ("conv.weight", "shared_MLP.0", "localization_fc1", "mlp.fc1")
    new = {}
    for k, v in sd.items():
        if k.startswith("atten_tps") or "norm" in k or k.startswith("TPE.localization_fc2"):
            continue
        if k.endswith("weight"):
            fan_in = int(np.prod(v.shape[1:]))
            bound = math.sqrt((6.0 if any(t in k for t in relu_fed) else 3.0) / fan_in)
            new[k] = torch.from_numpy(rs.uniform(-bound, bound, tuple(v.shape)).astype(np.float32))
        else:
            new[k] = torch.from_numpy(rs.uniform(-0.1, 0.1, tuple(v.shape)).astype(np.float32))
    new["TPE.localization_fc1.2.bias"] = new["TPE.localization_fc1.2.bias"] + 0.5
    for nm in ("norm1", "norm2"):
        new[f"TPE.atten.0.{nm}.weight"] = torch.from_numpy((1 + 0.1 * rs.standard_normal((16, 64))).astype(np.float32))
        new[f"TPE.atten.0.{nm}.bias"] = torch.from_numpy((0.1 * rs.standard_normal((16, 64))).astype(np.float32))
    new["TPE.localization_fc2.weight"] = torch.from_numpy((5e-5 * rs.standard_normal((64, 64))).astype(np.float32))
    bias = sd["TPE.localization_fc2.bias"].detach().cpu().view(32, 2).clone()
    xs, ys = bias[:, 0].clone(), bias[:, 1].clone()
    bias[:, 0] = (xs - 0.5) * 1.03 + 0.5 + 0.02 * (ys - 0.5)
    bias[:, 1] = ys + 0.04 * torch.sin(2 * math.pi * 1.3 * xs + 0.7)
    new["TPE.localization_fc2.bias"] = bias.view(-1)
    m.load_state_dict(new, strict=False)


# ----------------------------------------------------------------------------- BASELINE configs[3]
def _classical_inputs(F_, B, dev, seed):
    """img [B,3,64,256] ~ N(0,1); C' = the classical init lattice + a smooth per-image field (SURVEY 8d config 4)."""
    from tps_pp_b200 import constants as K
    inv, ph, _ = K.classical_tps_buffers(F_, (64, 256))
    base = torch.from_numpy(K.classical_init_bias(F_)).float()
    g = torch.Generator().manual_seed(seed)
    a = (torch.rand(B, 1, generator=g) - 0.5) * 0.2
    fr = 0.5 + 1.5 * torch.rand(B, 1, generator=g)
    phs = 6.2831853 * torch.rand(B, 1, generator=g)
    cp = base[None].repeat(B, 1, 1)
    cp[..., 1] = cp[..., 1] + a * torch.sin(fr * 3.14159265 * cp[..., 0] + phs)
    cp[..., 0] = cp[..., 0] * (1 + (torch.rand(B, 1, generator=g) - 0.5) * 0.1)
    gd = torch.Generator(device=dev).manual_seed(seed) if dev != "cpu" else g
    img = torch.randn((B, 3, 64, 256), device=dev, generator=gd)
    return img, cp.contiguous(), torch.from_numpy(inv), torch.from_numpy(ph)


def _classical_cpu(F_, steps, warmup, batch):
    """The reference's classical path on host cores: GridGenerator.build_P_prime (two bmm) + F.grid_sample
    (tps_preprocessor.py:72-83,270-282), restated in oracle/tpspp_oracle.py with the same torch CPU ops."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    img, cp, inv, ph = _classical_inputs(F_, batch, "cpu", 0)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            Bq = cp.shape[0]
            T_ = torch.bmm(inv[None].expand(Bq, -1, -1), torch.cat([cp, torch.zeros(Bq, 3, 2)], 1))
            grid = torch.bmm(ph[None].expand(Bq, -1, -1), T_).reshape(Bq, 64, 256, 2)
            torch.nn.functional.grid_sample(img, grid, padding_mode="border", align_corners=True)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    med = statistics.median(times)
    return batch / med, med * 1e3, cores


class _no_tf32_matmul:
    """cuBLAS fp32 without TF32 (the reference's numerics) for the library arm of a comparison."""

    def __enter__(self):
        self.prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False

    def __exit__(self, *exc):
        torch.backends.cuda.matmul.allow_tf32 = self.prev


def run_classical(args):
    """BASELINE configs[3]: high-res classical TPS rectification, 64x256x3 input, F = 20 / 40, batch 1024 per GPU: the
    fused grid generator + bilinear warp alone (the localisation network is not part of the north_star path)."""
    F_ = args.F
    B = args.batch
    workload = f"classical TPS warp (GridGenerator + grid_sample), 64x256x3 fp32, F={F_}, batch {B}/GPU (BASELINE configs[3])"
    rank, world, local = _dist_env()
    if args.impl == "reference":
        if rank != 0:
            return
        sb = min(B, 128)
        ips, ms, cores = _classical_cpu(F_, max(1, args.steps), max(0, args.warmup), sb)
        print(json.dumps({
            "impl": "reference", "metric": "classical_tps_rectified_img_per_s", "value": ips, "unit": "img/s", "n_gpus": args.gpus,
            "steps": max(1, args.steps), "warmup": max(0, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "global_batch": B, "sample": f"batch {sb} per step on host CPU, {cores} threads"},
            "cpu_baseline": {"value": ips, "unit": "img/s", "cores": cores, "kind": "port",
                             "sample": f"{max(1, args.steps)} steps of batch {sb} (median), torch CPU fp32 bmm + grid_sample, {cores} threads"},
            "e2e": {"value": ips, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)
        return
    import torch.distributed as dist
    from tps_pp_b200 import _native as N, functional as TF
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the TPS hot path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N.device_info()
    img, cp, inv, ph = _classical_inputs(F_, B, dev, 1234 + rank)
    cp, inv, ph = cp.to(dev), inv.to(dev), ph.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(src):
        return TF.tps_warp(src, None, cp, None, ph, None, inv, (64, 256), mode=N.MODE_CLASSICAL, theta=0.0)[0]

    launches = 0
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            step(img)
        barrier()
        sampler = ClockSampler(local)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            out = step(img)
            launches += N.last_launch_count()
        e1.record()
        barrier()
        clocks = sampler.stop()
        total_ms = e0.elapsed_time(e1)
        if args.dump_outputs and rank == 0:
            _dump_outputs(args.dump_outputs, {"output": out})
        del out
        # end to end with host buffers: H2D of the images + control points, D2H of the rectified images, every step
        himg, hcp = img.cpu().pin_memory(), cp.cpu().pin_memory()
        hout = torch.empty_like(himg).pin_memory()
        dimg = [torch.empty_like(img) for _ in range(2)]
        s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]

        def e2e_run(nsteps):
            for k in range(2):
                ev_free[k].record(main)
            for i in range(nsteps):
                k = i & 1
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_free[k])
                    dimg[k].copy_(himg, non_blocking=True)
                    cp.copy_(hcp, non_blocking=True)
                    ev_in[k].record(s_in)
                main.wait_event(ev_in[k])
                r = step(dimg[k])
                ev_done[k].record(main); ev_free[k].record(main)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_done[k])
                    hout.copy_(r, non_blocking=True)
                r.record_stream(s_out)
            main.wait_stream(s_out)

        e2e_run(2)
        barrier()
        e2e_steps = max(3, min(args.steps, 8))
        reps = []
        for _ in range(3):        # median of three repetitions: 400 MB of pinned-memory traffic per step is at the mercy of the host
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            e2e_run(e2e_steps)
            f1.record()
            barrier()
            reps.append(f0.elapsed_time(f1))
        e2e_ms = sorted(reps)[1]
    # the whole drop-in module (SURVEY 8f rank 4): TPSPreprocessor.forward = localisation network + the warp above, device-
    # resident images, with the native localisation network (tpspp_locnet_fwd) and with the cuDNN / cuBLAS fp32 stack
    module = None
    if rank == 0 and world == 1:
        import tps_pp_b200 as T
        torch.manual_seed(0)
        tp = T.TPSPreprocessor(num_fiducial=F_, img_size=(64, 256), rectified_img_size=(64, 256), num_img_channel=3).to(dev).eval()
        module = {"what": "TPSPreprocessor.forward(img[B,3,64,256]) = LocalizationNetwork (1.87 GFLOP/img) + GridGenerator + grid_sample, "
                          "device-resident images, random-init weights, eval mode"}
        with torch.no_grad(), torch.backends.cudnn.flags(enabled=True, allow_tf32=False), _no_tf32_matmul():
            for impl, nst in (("auto", 5), ("library", 3)):
                tp.locnet_impl = impl
                for _ in range(2):
                    tp(img)
                torch.cuda.synchronize()
                m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                m0.record()
                for _ in range(nst):
                    tp(img)
                m1.record()
                torch.cuda.synchronize()
                ms = m0.elapsed_time(m1) / nst
                name = "native" if impl == "auto" else "library"
                module[name + "_locnet_ms_per_step"] = ms
                module[name + "_locnet_img_per_s"] = B / (ms * 1e-3)
                if impl == "auto":
                    module["locnet_native"] = bool(tp._last_locnet_native)
    t = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = (float(v) for v in t.tolist())
    step_ms = total_ms / args.steps
    peak, peak_src = _peaks()
    # SURVEY 8(d): 2 * C*H*W*4 + 8F bytes per image; constants (P_hat [n, F+3], inv_delta_C) once per launch
    bytes_launch = B * (2 * 3 * 64 * 256 * 4 + 8 * F_) + 16384 * (F_ + 3) * 4 + (F_ + 3) ** 2 * 4
    achieved = bytes_launch / (step_ms * 1e-3) / 1e9
    dfma = B * 16384 * (F_ + 3) * 2                       # fp64 FMAs of grid = P_hat . T per launch
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ips, ms, cores = _classical_cpu(F_, 5, 1, 128)
        cpu = {"value": ips, "unit": "img/s", "cores": cores, "kind": "port",
               "sample": f"5 steps of batch 128 (median {ms:.0f} ms), torch CPU fp32 bmm + grid_sample, {cores} threads"}
    if rank == 0:
        print(json.dumps({
            "metric": "classical_tps_rectified_img_per_s", "value": world * B * args.steps / (total_ms * 1e-3), "unit": "img/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 pixels / f64 grid", "data": "synthetic",
            "config": {"workload": workload, "global_batch": world * B, "parallelism": f"batch-shard x{world}, no collective",
                       "l2": f"images {B * 3 * 64 * 256 * 4 >> 20} MB/step > 126 MB L2 (no flush needed)"},
            "roofline": {"kernel": "classical_T_kernel + warp_fwd_classical_tiled_kernel (timed together: the step is these two launches)",
                         "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "peak_source": peak_src, "bytes_per_launch": bytes_launch, "avg_launch_ms": step_ms,
                         "fp64_fma_per_launch": dfma,
                         "note": "the grid P_hat.T is evaluated in fp64 (pixel parity 1e-5 needs coordinates to ~1e-8): "
                                 f"{dfma / 1e9:.2f} G DFMA per launch is a second floor next to the HBM one"},
            "cpu_baseline": cpu, "module": module,
            "e2e": {"value": world * B * e2e_steps / (e2e_ms * 1e-3), "unit": "img/s", "h2d_bytes_per_step": himg.numel() * 4 + hcp.numel() * 4,
                    "d2h_bytes_per_step": hout.numel() * 4, "steps": e2e_steps, "repetitions": "median of 3"},
            "gpu_launches": launches, "clocks": clocks}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU,
                    help="images per GPU (default = BASELINE configs[1]; 1024 = the per-GPU shard of config 5 at 8 GPUs)")
    ap.add_argument("--workload", default="tps_pp", choices=["tps_pp", "classical64x256"],
                    help="tps_pp = BASELINE configs[1] (default, the headline line); classical64x256 = configs[3], the high-res "
                         "classical TPS warp (64x256x3 images, batch 1024, --F 20|40 control points)")
    ap.add_argument("--F", type=int, default=20, choices=[20, 40], help="control points of the classical64x256 workload")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="BASELINE configs[4]: split this many images over the ranks (strong scaling, e.g. 8192) instead of "
                         "--batch per GPU (weak scaling)")
    ap.add_argument("--head", default="tc", choices=["tc", "tc3x", "fp32", "bf16", "library"],
                    help="head arithmetic: tcgen05 split-fp32 (default, fp32-level accuracy; tc3x = all-tf32 3xTF32 convs), CUDA-core fp32, "
                         "tcgen05 with bf16 conv operands (reduced precision, reported separately), or "
                         "cuDNN/cuBLAS library ops")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (rank 0's shard) to DIR/<name>.npy as float32; "
                         "above 64 MB in all, the same seeded sample of images is kept from every array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    if args.workload == "classical64x256":
        if args.batch == BATCH_PER_GPU:
            args.batch = 1024
        run_classical(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
