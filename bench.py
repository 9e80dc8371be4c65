#!/usr/bin/env python
"""bench.py -- ResNet-18 TQ (g=8, alpha=12) inference throughput on B200, with the TR-encode
kernel's HBM roofline and the reference's CPU path timed beside it.

    python bench.py --gpus N --steps K --warmup W            # this repo (one rank per GPU)
    python bench.py --impl reference --gpus N --steps K ...  # reference CPU path (rank 0 only)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's logits to DIR

A step = one forward of the term-quantised ResNet-18 over one synthetic batch of 256 images
per GPU (BASELINE.json configs[1]; reference setting evaluate_group_size.py:71-74: 9-bit
weights/activations, g=8, alpha=12, data_terms=3; first conv unwrapped).  Weak scaling: every
rank runs its own 256 images and the logits are all-gathered (NCCL) inside the step.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

SETTING = dict(weight_bits=9, group_size=8, weight_terms=12, data_bits=9, data_terms=3)
BATCH = 256
METRIC = "resnet18_tq_g8_a12_images_per_sec"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}

    def __init__(self, index, period=0.02):
        # NVML queries serialise on a driver-wide lock: 8 ranks polling at 100 Hz cost 0.28 ms per 2.1 ms step
        # (measured, DESIGN.md section 7), so only rank 0 samples, at 50 Hz
        super().__init__(daemon=True)
        self.period = period
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        while self.nv is not None and not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def sample_now(self):
        """One sample from the calling thread (used while the GPU drains the enqueued timed region)."""
        if self.nv is None:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            mask = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, name in self.REASONS.items():
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_mhz_min": s[0] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------------
def build_tq_resnet18(device):
    from torchvision.models import resnet18
    from term_quantization_b200 import cnn_models
    torch.manual_seed(0)
    model = resnet18(weights=None).eval().to(device)
    params = cnn_models.static_conv_layer_settings(model, SETTING["weight_bits"], SETTING["group_size"],
                                                   SETTING["weight_terms"])
    qmodel = cnn_models.convert_model(model, params, SETTING["data_bits"], SETTING["data_terms"])
    return qmodel.eval()


class KernelTimer:
    """Wraps the Python entry points of this repo's kernels so that every launch inside the
    timed region is bracketed by CUDA events on the launching stream: per-launch durations and
    algorithmic bytes / flops for the roofline objects."""

    def __init__(self):
        from term_quantization_b200 import conv_codes, tr_cuda
        self.on = False
        self.records = {"tr_encode": [], "conv": [], "stem": [], "pool": []}
        self.targets = [(tr_cuda, "tr", "tr_encode", lambda a, k, out: a[0].numel() * a[0].element_size() * 2),
                        (tr_cuda, "tr_codes", "tr_encode",
                         lambda a, k, out: a[0].numel() * (a[0].element_size() + out.element_size())),
                        (conv_codes, "conv2d_codes", "conv",
                         lambda a, k, out: 2 * out.numel() * a[1].shape[0] * a[1].shape[2]),
                        (conv_codes, "conv2d_codes_fused", "conv",
                         lambda a, k, out: (2 * (out[0] if out[0] is not None else out[1]).numel()
                                            * a[1].shape[0] * a[1].shape[2],
                                            # algorithmic bytes of this launch: codes in, weights in, residual in,
                                            # fp32 tile out, code tile out -- each tensor once
                                            a[0].numel() * 2 + a[1].numel() * 2
                                            + (k["residual"].numel() * 4 if k.get("residual") is not None else 0)
                                            + (out[0].numel() * 4 if out[0] is not None else 0)
                                            + (out[1].numel() * 2 if out[1] is not None else 0))),
                        (conv_codes, "stem_conv7x7s2", "stem", lambda a, k, out: 2 * out[0].numel() * 147),
                        (conv_codes, "stem_conv_pool", "stem", lambda a, k, out: 2 * out[0].numel() * 4 * 147),
                        (conv_codes, "bn_relu_maxpool_encode", "pool",
                         lambda a, k, out: a[0].numel() * 4 + out[0].numel() * 4
                         + (out[1].numel() * 2 if out[1] is not None else 0))]
        self.saved = []

    def __enter__(self):
        for mod, attr, key, work in self.targets:
            orig = getattr(mod, attr)
            self.saved.append((mod, attr, orig))

            def timed(*a, _orig=orig, _key=key, _work=work, **k):
                if not self.on:
                    return _orig(*a, **k)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = _orig(*a, **k)
                e1.record()
                w = _work(a, k, out)
                self.records[_key].append((e0, e1) + (w if isinstance(w, tuple) else (w, 0)))
                return out
            setattr(mod, attr, timed)
        return self

    def __exit__(self, *exc):
        for mod, attr, orig in self.saved:
            setattr(mod, attr, orig)

    def summary(self, key):
        rec = self.records[key]
        return len(rec), sum(r[2] for r in rec), sum(r[0].elapsed_time(r[1]) for r in rec)

    def bytes(self, key):
        return sum(r[3] for r in self.records[key])


def ncu_conv_traffic():
    """DRAM bytes per launch of the conv kernel from this round's ncu capture (profiles/r02_conv_traffic.json, written
    by tools/ncu_traffic.py from `ncu --set full` of this same command) -- used only while the kernel source it was
    taken from is unchanged (sha256 of csrc/tq_gemm.cu); otherwise null rather than a stale number."""
    import hashlib
    try:
        with open(os.path.join(ROOT, "profiles", "r02_conv_traffic.json")) as f:
            rec = json.load(f)
        src = os.path.join(ROOT, "term_quantization_b200", "csrc", "tq_gemm.cu")
        if hashlib.sha256(open(src, "rb").read()).hexdigest() != rec["tq_gemm_cu_sha256"]:
            return None, "profiles/r02_conv_traffic.json is from an older tq_gemm.cu: not used"
        return float(rec["dram_bytes_per_launch"]), "profiles/r02_conv_traffic.json (" + rec.get("how", "ncu --set full") + ")"
    except Exception:
        return None, None


def tr_encode_roofline(dev, peak, peak_src, iters=20):
    """BASELINE metric 1: TR-encode GB/s at the largest ResNet-18 activation (256x64x56x56 fp32,
    g=1, 9-bit, 3 terms, drop-in fp32 -> fp32 contract: 8 B/element).  Two 205 MB inputs rotate
    (> 126 MB L2); every launch is timed with CUDA events on its stream."""
    from term_quantization_b200 import tr_cuda
    n = 256 * 64 * 56 * 56
    g = torch.Generator(device=dev).manual_seed(7)
    xs = [torch.relu(torch.randn(1, n, 1, 1, device=dev, generator=g)) for _ in range(2)]
    out = torch.empty_like(xs[0])
    sf = float(xs[0].max()) / 512
    for i in range(3):
        tr_cuda.tr(xs[i % 2], sf, 9, 1, 3, out=out)
    torch.cuda.synchronize()
    evs = []
    for i in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tr_cuda.tr(xs[i % 2], sf, 9, 1, 3, out=out)
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in evs) / iters
    ach = n * 8 / (ms * 1e-3) / 1e9
    return {"kernel": "tq::tr_elem_kernel<float,float> on 51,380,224 elements (ResNet-18 layer1 activation at "
                      "batch 256), g=1, 9-bit, 3 terms", "bound": "hbm", "achieved": ach, "peak": peak,
            "unit": "GB/s", "frac": ach / peak, "frac_of_nominal_8000": ach / 8000.0, "traffic": None,
            "peak_source": peak_src, "launches_timed": iters, "algorithmic_bytes_per_launch": n * 8,
            "ms_per_launch": ms}


def run_b200(args):
    from term_quantization_b200 import _lib, inference
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = inference.bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # fp32 convs must be true fp32 for the 1e-5 logit tolerance (TF32 keeps 10 mantissa bits)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True

    model = build_tq_resnet18(dev)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    nbuf = 2
    # images travel and are stored as bf16 (BASELINE.json configs[1]: "bf16 -> int8"): synthetic randn
    # rounded to bf16; --input-dtype fp32 keeps the reference loader's fp32 tensors
    in_dtype = torch.bfloat16 if (args.input_dtype == "bf16" and args.conv_backend == "fused") else torch.float32
    images = [torch.randn(BATCH, 3, 224, 224, device=dev, generator=gen).bfloat16().float() for _ in range(nbuf)]
    inference.calibrate(model, [images[0][:64]])          # untimed: histograms + fused sweep
    engines = {}
    if args.conv_backend in ("tcgen05", "fused"):
        from term_quantization_b200 import fused, tr_layer
        model = model.to(memory_format=torch.channels_last)
        images = [im.contiguous(memory_format=torch.channels_last) for im in images]
        if args.conv_backend == "tcgen05":
            switched, skipped = tr_layer.use_tensor_cores(model, engine=args.conv_engine)
            assert len(switched) == 19 and not skipped, (switched, skipped)
        if args.conv_backend == "fused":
            model = fused.FusedResNet(model, stem=args.stem, engine=args.conv_engine)
            for blk in model.blocks:
                for c in blk:
                    if c is not None:
                        k = f"{c.plan.engine} x{c.plan.groups}" if c.plan.engine == "f16" else f"i8 {c.plan.planes_w}w-plane"
                        engines[k] = engines.get(k, 0) + 1
    images = [im.to(in_dtype) for im in images]
    use_graphs = args.conv_backend == "fused" and not args.no_cuda_graphs
    runner = inference.ShardedInference(model, dev, cuda_graphs=use_graphs, gather=args.gather)
    eager = inference.ShardedInference(model, dev, gather=args.gather) if use_graphs else runner

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM ----------------------------------------------------
    for i in range(args.warmup):
        runner.forward(images[i % nbuf])
    runner.finish()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.profiler.start()          # no-op unless ncu runs with --profile-from-start off
    e0.record()
    for i in range(args.steps):
        out = runner.forward(images[i % nbuf])
    fin = runner.finish()                # outstanding / final gather of logits: inside the timed region
    e1.record()
    if rank == 0:
        sampler.sample_now()             # the GPU is still draining the region: at least one sample under load
    barrier()
    torch.cuda.profiler.stop()
    ms_total = e0.elapsed_time(e1)
    out = (fin[-1] if (fin is not None and fin.dim() == 3) else (fin if fin is not None else out)).clone()
    # the same K steps again, launch by launch with CUDA events around every kernel of this repo (the
    # headline region above runs without them: as CUDA-graph replays when enabled): per-kernel durations
    # for the roofline objects and the launch count
    for i in range(args.warmup if use_graphs else 0):      # the eager path's own warm-up (allocator pools)
        eager.forward(images[i % nbuf])
    eager.finish()
    barrier()
    with KernelTimer() as trt:
        trt.on = True
        launches0 = _lib.launch_count()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for i in range(args.steps):
            eager.forward(images[i % nbuf])
        eager.finish()
        k1.record()
        barrier()
        launches = _lib.launch_count() - launches0
        trt.on = False
        ms_instrumented = k0.elapsed_time(k1)
        n_tr, tr_bytes, tr_ms = trt.summary("tr_encode")
        n_cv, cv_flops, cv_ms = trt.summary("conv")
        n_st, st_flops, st_ms = trt.summary("stem")
        n_pl, pl_bytes, pl_ms = trt.summary("pool")
    clocks = sampler.finish()
    diag = None
    if args.diag:
        # extra timed loops (no clock sampler running): graph replay vs eager launches, same K steps
        def timed_loop(r):
            for i in range(3):
                r.forward(images[i % nbuf])
            r.finish()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(args.steps):
                r.forward(images[i % nbuf])
            r.finish()
            b.record()
            barrier()
            tt = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item()) / args.steps
        diag = {"graph_no_sampler_ms": timed_loop(runner), "eager_no_sampler_ms": timed_loop(eager)}
        nogather = inference.ShardedInference(model, dev, cuda_graphs=use_graphs, gather="end")
        t_ng = timed_loop(nogather)
        diag["graph_gather_end_ms"] = t_ng
    per_rank = None
    if world > 1:
        # every rank's own view: its timed region, its clocks, its kernel time (the last is independent of
        # the per-step synchronisation with the other ranks)
        mine = {"rank": rank, "ms_per_step": ms_total / args.steps, "sm_mhz": clocks["sm_mhz"],
                "sm_mhz_min": clocks.get("sm_mhz_min"), "reasons": clocks["reasons"],
                "conv_kernels_ms_per_step": cv_ms / args.steps,
                "instrumented_ms_per_step": ms_instrumented / args.steps}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    assert out.shape == (BATCH * world, 1000) and bool(torch.isfinite(out).all())

    # ---- e2e: pinned host images -> H2D -> forward -> all-gather -> logits D2H -------------
    host = [torch.randn(BATCH, 3, 224, 224).bfloat16().float() for _ in range(2)]
    if args.conv_backend in ("tcgen05", "fused"):
        host = [h.contiguous(memory_format=torch.channels_last) for h in host]
    host = [h.to(in_dtype).pin_memory() for h in host]
    # three device slots: the copies of shards i+1 and i+2 are in flight while forward i runs
    s0 = runner.stage(host[0])
    s1 = runner.stage(host[1])
    for i in range(max(args.warmup, 1)):
        nxt = runner.stage(host[i % 2])
        runner.run(s0)
        s0, s1 = s1, nxt
    runner.finish()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        nxt = runner.stage(host[i % 2])
        host_logits = runner.run(s0)
        s0, s1 = s1, nxt
    runner.finish()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    assert bool(torch.isfinite(host_logits).all())
    # ---- e2e with uint8 images: 1 byte per value over PCIe, ToTensor + Normalize on the device --------------------
    e2e_u8 = None
    if args.conv_backend == "fused" and not args.no_e2e_uint8:
        front = inference.U8Frontend(model)
        runner8 = inference.ShardedInference(front, dev, cuda_graphs=use_graphs, gather=args.gather)
        host8 = [torch.randint(0, 256, (BATCH, 224, 224, 3), dtype=torch.uint8).pin_memory() for _ in range(2)]
        a0 = runner8.stage(host8[0])
        a1 = runner8.stage(host8[1])
        for i in range(max(args.warmup, 3)):
            nxt = runner8.stage(host8[i % 2])
            runner8.run(a0)
            a0, a1 = a1, nxt
        runner8.finish()
        barrier()
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record()
        for i in range(args.steps):
            nxt = runner8.stage(host8[i % 2])
            host_logits8 = runner8.run(a0)
            a0, a1 = a1, nxt
        runner8.finish()
        u1.record()
        barrier()
        t = torch.tensor([u0.elapsed_time(u1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        assert bool(torch.isfinite(host_logits8).all())
        e2e_u8 = {"value": BATCH * world * args.steps / (float(t.item()) * 1e-3), "unit": "images/s",
                  "ms_per_step": float(t.item()) / args.steps,
                  "h2d_bytes_per_step": BATCH * 224 * 224 * 3 * world, "d2h_bytes_per_step": int(host_logits8.numel()) * 4 * world,
                  "note": "same engine fed uint8 NHWC images; ((u8 / 255) - mean) / std as the reference loader computes it "
                          "(util.py:12-27), rounded to the bf16 the engine consumes, inside the stem's fold pass on the device "
                          "(tq_stem_conv7x7s2_u8; the same values as tq_u8_normalize_bf16)"}
        del runner8, front
    # what the box allows: the same host -> device copies alone, all ranks at once (max over ranks)
    import bench_extra
    barrier()
    t = torch.tensor([bench_extra.h2d_ceiling(host, [b for b in runner._stage if b is not None], args.steps, runner.copy_stream)],
                     dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    h2d_only_ms = float(t.item())
    barrier()

    line = None
    if rank == 0:
        peak, peak_src = peaks()
        ach = tr_bytes / (tr_ms * 1e-3) / 1e9 if tr_ms > 0 else 0.0
        tr_roof = {"kernel": "tq::tr_elem_kernel (g=1 TR encode; standalone launches only -- in the fused "
                             "engine all but the first encode run inside the conv epilogue; fp32 in, " + ("fp16 codes out: 6 B/elem" if args.conv_backend != "cudnn_fp32"
                                                         else "fp32 out: 8 B/elem") + ")",
                   "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                   "traffic": None, "peak_source": peak_src, "launches_timed": n_tr,
                   "algorithmic_bytes": tr_bytes, "kernel_ms_total": tr_ms, "share_of_step": tr_ms / ms_instrumented}
        conv_roof = None
        if n_cv:
            try:
                with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                    pk = json.load(f)
                # each conv launch is timed alone with CUDA events and the whole pass lasts tens of ms at full clocks:
                # the applicable ceiling is the BURST figure
                tpeak, tsrc = float(pk["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst; kind::f16 runs at the bf16 rate)"
                tsus = float(pk.get("bf16_tflops_sustained", 0)) or None
            except Exception:
                tpeak, tsrc, tsus = 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s burst)", 1400.0
            tach = cv_flops / (cv_ms * 1e-3) / 1e12
            traffic, traffic_src = ncu_conv_traffic()
            conv_roof = {"kernel": "tq::conv_igemm_kernel (tcgen05 implicit GEMM on term codes, exact int32 accumulators, fused "
                                   "BN/residual/ReLU/encode epilogue, 19 launches per forward)",
                         "bound": "tensor", "achieved": tach, "peak": tpeak, "unit": "TFLOP/s", "frac": tach / tpeak,
                         "frac_of_sustained": (tach / tsus) if tsus else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": trt.bytes("conv") / n_cv,
                         "algorithmic_bytes_model": "per launch, from the launch's own tensor shapes: fp16 codes in + fp16 weight codes "
                                                    "+ fp32 residual in + fp32 tile out + fp16 codes out, each once",
                         "peak_source": tsrc, "launches_timed": n_cv,
                         "algorithmic_flops": cv_flops, "kernel_ms_total": cv_ms, "share_of_step": cv_ms / ms_instrumented,
                         "whole_step_TFLOPs": (cv_flops + st_flops) / args.steps / (ms_total / args.steps * 1e-3) / 1e12,
                         "timed": "CUDA events around each launch in an eager pass of the same K steps"}
        dominant, other = (conv_roof, tr_roof) if (conv_roof and cv_ms > tr_ms) else (tr_roof, conv_roof)
        if other is tr_roof and n_tr == 0:
            other = None            # fused engine: every encode runs inside a conv / stem epilogue (see "tr_encode")
        line = {
            "metric": METRIC, "value": BATCH * world * args.steps / (ms_total * 1e-3),
            "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": ("int term codes (TR encode) -> exact int32 accumulators on tcgen05 (kind::f16 with statically "
                                       "proven fp32 K-chunk accumulators summed in int32, or kind::i8 planes with s32 accumulators)"
                                       if args.conv_backend != "cudnn_fp32" else "f32 values (TR encode); f32 conv"),
            "data": "synthetic (randn images rounded to bf16, random-init torchvision resnet18, seed 0)",
            "config": {"workload": "ResNet-18 TQ inference, batch 256 per GPU at 3x224x224 "
                                   "(BASELINE.json configs[1])", **SETTING,
                       "global_batch": BATCH * world, "parallelism": (f"batch-sharded x{world}, logits all-gather (NCCL) " + {
                           "step": "every step on the compute stream", "async": "every step on a side stream",
                           "end": "once, after the last step (inside the timed region)"}[args.gather])
                       if world > 1 else "single GPU",
                       "conv_backend": args.conv_backend, "conv_engine": args.conv_engine, "engines_per_layer": engines,
                       "input_dtype": str(in_dtype).replace("torch.", ""),
                       "cuda_graphs": bool(use_graphs),
                       "numa": (f"rank pinned to the {len(numa_cpus)} CPUs local to its GPU" if numa_cpus else "not pinned"),
                       "l2": "activations per step (2.08 GB fp32 through TR) exceed the 126 MB L2; "
                             "input batches rotate between 2 buffers"},
            "e2e": {"value": BATCH * world * args.steps / (e2e_ms * 1e-3), "unit": "images/s",
                    "h2d_bytes_per_step": BATCH * 3 * 224 * 224 * host[0].element_size() * world,
                    "d2h_bytes_per_step": int(host_logits.numel()) * 4 * world,
                    "ms_per_step": e2e_ms / args.steps,
                    "note": "bytes are job totals per step (each rank copies its own 256-image shard in and its own "
                            "logits out; the gathered logits stay on the devices); 3 staging slots per rank",
                    "h2d_only_ms_per_step": h2d_only_ms,
                    "h2d_ceiling_gbs": BATCH * 3 * 224 * 224 * host[0].element_size() * world / (h2d_only_ms * 1e-3) / 1e9,
                    "h2d_ceiling_images_per_s": BATCH * world / (h2d_only_ms * 1e-3),
                    "h2d_ceiling_note": "the same pinned-host -> device copies with no compute, all ranks at once, max over ranks: "
                                        "the e2e number cannot exceed this on this box"},
            **({"e2e_uint8": e2e_u8} if e2e_u8 else {}),
            "gpu_launches": int(launches),
            "clocks": clocks,
            **({"per_rank": per_rank} if per_rank else {}),
            **({"diag": diag} if diag else {}),
            "roofline": dominant,
            "roofline_other": other,
            "tr_encode": tr_encode_roofline(dev, peak, peak_src),
            "kernel_ms_per_step": {
                "note": "CUDA-event time per step of each kernel family in the instrumented eager pass",
                "conv_igemm_wrapped_convs": cv_ms / args.steps, "conv_igemm_launches_per_step": n_cv // args.steps,
                "stem_prepare_plus_conv_igemm_stem_with_fused_pool": st_ms / args.steps,
                "bn_relu_maxpool_encode": pl_ms / args.steps,
                "bn_relu_maxpool_encode_GBs": (pl_bytes / (pl_ms * 1e-3) / 1e9) if pl_ms > 0 else None,
                "tr_elem_standalone": tr_ms / args.steps, "instrumented_step": ms_instrumented / args.steps},
        }
        if world == 1 and not args.no_extras:
            # BASELINE.md section 3's grid and the other BASELINE configs, after every headline region; the big buffers of
            # the headline run are released first
            del runner, eager, images
            torch.cuda.empty_cache()
            grid, beat = bench_extra.tr_grid(dev, peak, with_ref=not args.no_cpu_baseline)
            line["tr_grid"] = grid
            line["kernel_to_beat"] = {"what": "the reference's own kernel (kernels/tr_cuda_kernel.cu:58-125, byte-identical body, "
                                              "recompiled for sm_100a: oracle/_ref/libtq_ref_gpu.so) on the same tensors, same timing",
                                      "rows": beat} if beat else None
            line["other_configs"] = bench_extra.other_configs(dev)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_reference_images_per_sec(sample_batch=args.cpu_batch, steps=1)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": out})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def dump_outputs(directory, arrays):
    """Writes each tensor as DIR/<name>.npy (float32) so that two builds run with the same arguments, and hence the
    same seeded inputs, can be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------
# reference arm: the reference's module stack on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_reference_images_per_sec(sample_batch, steps, warmup=0):
    """Times the reference stack (oracle/ref_stack.py: reference kernel body on the host for TR,
    PyTorch CPU fp32 convs) on a bounded sample of the same workload."""
    from torchvision.models import resnet18
    from oracle import ref_stack, tq_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = resnet18(weights=None).eval()
    t0 = time.time()
    q = ref_stack.convert_cnn(model, SETTING["weight_bits"], SETTING["group_size"], SETTING["weight_terms"],
                              SETTING["data_bits"], SETTING["data_terms"])
    convert_s = time.time() - t0
    x = torch.randn(sample_batch, 3, 224, 224, generator=torch.Generator().manual_seed(1234)).bfloat16().float()
    # timing-only scale factors (max/2^bits of a tracking pass); logit parity is tested in tests/
    maxes = []

    def grab(mod, inp):
        maxes.append(float(inp[0].abs().max()))
    hs = [m.register_forward_pre_hook(grab) for m in ref_stack.quantizers(q)]
    with torch.no_grad():
        q(x[:2])
    for h in hs:
        h.remove()
    ref_stack.set_scale_factors(q, [max(m, 1e-6) / 2 ** SETTING["data_bits"] for m in maxes])
    with torch.no_grad():
        for _ in range(warmup):
            q(x)
        t0 = time.time()
        for _ in range(steps):
            q(x)
        dt = time.time() - t0
    return {"value": sample_batch * steps / dt, "unit": "images/s", "cores": cores,
            "kind": "reference" if O.have_ref() else "port",
            "sample": f"{steps} forward(s) of batch {sample_batch} (of the 256-image step), TR via "
                      f"{'oracle/_ref (reference kernel body on host)' if O.have_ref() else 'oracle port'}"
                      f" on {cores} threads + torch CPU fp32 conv; weight conversion {convert_s:.1f}s untimed",
            "seconds": dt}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    world = int(os.environ.get("WORLD_SIZE", "1"))
    base = cpu_reference_images_per_sec(sample_batch=args.cpu_batch, steps=args.steps, warmup=min(args.warmup, 1))
    v = base["value"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * args.cpu_batch / v,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (randn images rounded to bf16, random-init torchvision resnet18, seed 0)",
            "config": {"workload": "ResNet-18 TQ inference, batch 256 per GPU at 3x224x224 "
                                   "(BASELINE.json configs[1])", **SETTING,
                       "note": f"each step is a bounded sample: batch {args.cpu_batch} on the host cores"},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--conv-backend", default="fused", choices=["fused", "tcgen05", "cudnn_fp32"],
                    help="fused: code-domain tcgen05 convs with BN/residual/ReLU/next-layer encode in the "
                         "epilogue (fused.FusedResNet); tcgen05: same kernel layer by layer under the "
                         "unchanged torchvision graph; cudnn_fp32: the reference's float path")
    ap.add_argument("--input-dtype", default="bf16", choices=["bf16", "fp32"],
                    help="dtype of the image batches in HBM and over PCIe (fused engine; bf16 per BASELINE configs[1])")
    ap.add_argument("--stem", default="tcgen05", choices=["tcgen05", "tcgen05_pool", "cudnn"],
                    help="fused engine: two-launch tensor-core stem, one-kernel stem (pooling in the conv epilogue), cuDNN")
    ap.add_argument("--gather", default="step", choices=["step", "async", "end"],
                    help="when the other ranks' logits are collected (inference.ShardedInference)")
    ap.add_argument("--diag", action="store_true", help="extra timed loops: graph vs eager, no clock sampler")
    ap.add_argument("--no-cuda-graphs", action="store_true", help="launch the forward kernel by kernel")
    ap.add_argument("--cpu-batch", type=int, default=16, help="images per CPU-baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip tr_grid / kernel_to_beat / other_configs")
    ap.add_argument("--no-e2e-uint8", action="store_true", help="skip the additional end-to-end measurement with uint8 images")
    ap.add_argument("--conv-engine", default="auto", choices=["auto", "f16", "i8"],
                    help="how the exact accumulator is obtained per layer (conv_codes.plan_weight): auto = kind::f16 where "
                         "proven from the weights, kind::i8 planes otherwise")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the logits of the last one (the gathered logits of the whole "
                         "job, float32) to DIR/logits.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path; --impl reference times a CPU sample instead")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    # stdout carries ONE JSON line: anything a library prints to file descriptor 1 meanwhile (NCCL's version banner,
    # for one) goes to stderr; the descriptor is restored for the final print
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        if args.impl == "reference":
            line = run_reference(args)
        else:
            line = run_b200(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
