"""ResNet-50 TQ (9-bit weights, g = 8, alpha = 12, 3 data terms) at batch 256 on one GPU: fused.FusedResNet against the
layer-by-layer tcgen05 path and the reference's float path.

The model is random-init with randomised BatchNorm statistics, calibrated on 16 of the images; the images are bf16 in
HBM (the float and tcgen05 paths read them as fp32, as the reference's loader hands them over).  Each path is captured as
one CUDA graph and the three are replayed in alternation, round after round, in one process with TF32 off; per path the
median and the spread (min, max) of the per-round times, images/s and the wrapped convs' TFLOP/s (2 * MACs of the 52
wrapped convs, computed from the layer shapes here).  Also written: the exact engine and accumulator groups of every
fused conv, the fused logits against the tcgen05 path's, and the kernels of one eager fused forward (torch.profiler).
The card's name, power limit and max SM clock are read in the same run.

Usage: python tools/resnet_bench.py [--out profiles/r09_resnet50_bench.json] [--rounds 15] [--replays 5]
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from term_quantization_b200 import cnn_models, fused, inference, tr_layer  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, check=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = (v.strip() for v in line.split(","))
        return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}
    except Exception as e:                                   # reported, never guessed
        return {"error": f"nvidia-smi query failed: {e}"}


def randomise_bn(model, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for mod in model.modules():
            if isinstance(mod, nn.BatchNorm2d):
                n = mod.num_features
                mod.running_mean.copy_(torch.randn(n, device="cuda", generator=g) * 0.2)
                mod.running_var.copy_(torch.rand(n, device="cuda", generator=g) + 0.5)
                mod.weight.copy_(torch.rand(n, device="cuda", generator=g) + 0.5)
                mod.bias.copy_(torch.randn(n, device="cuda", generator=g) * 0.2)


def wrapped_macs(model, hw):
    """MACs per image of every conv but the first (the wrapped ones), from the output shapes of one forward."""
    macs = []

    def hook(mod, inp, out):
        kh, kw = mod.weight.shape[2:]
        macs.append(out[0].nelement() * (mod.in_channels // mod.groups) * kh * kw)
    hs = [c.register_forward_hook(hook) for c in model.modules() if type(c) is nn.Conv2d]
    with torch.no_grad():
        model(torch.zeros(1, 3, hw, hw, device="cuda"))
    for h in hs:
        h.remove()
    return sum(macs[1:])


def capture(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    return graph, out


def time_replays(graph, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def layer_plan(f):
    """(name, K, Cout, stride, engine, accumulator groups) of every fused conv, in launch order per block."""
    names = []
    for si, stage in enumerate((f.model.layer1, f.model.layer2, f.model.layer3, f.model.layer4)):
        for bi, _ in enumerate(stage):
            names.append([f"layer{si + 1}.{bi}.conv{k}" for k in (1, 2, 3)] + [f"layer{si + 1}.{bi}.downsample.0"])
    out = []
    for blk, nm in zip(f.blocks, names):
        for c, n in zip(blk, nm[:len(blk) - 1] + nm[-1:]):
            if c is not None:
                RS, Cout, C = c.w.shape
                out.append({"layer": n, "K": RS * C, "cout": Cout, "stride": c.stride, "engine": c.plan.engine,
                            "groups": c.plan.groups})
    return out


def eager_split(f, x):
    """Kernels of one eager fused forward, in launch order (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with torch.no_grad():
        f(x)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            f(x)
            torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
    launches = [{"kernel": e.name[:120], "us": round(e.time_range.elapsed_us(), 2)} for e in kernels]
    return {"launches": launches, "n_launches": len(launches), "sum_us": round(sum(k["us"] for k in launches), 1)}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_resnet50_bench.json"))
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--replays", type=int, default=5, help="graph replays per path per round")
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("resnet_bench needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.set_device(0)
    info = gpu_info()
    import torchvision
    torch.manual_seed(0)
    base = torchvision.models.resnet50(weights=None).cuda().eval()
    randomise_bn(base)
    macs = wrapped_macs(base, 224)
    q = cnn_models.convert_model(base, cnn_models.static_conv_layer_settings(base, 9, 8, 12), 9, 3)
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(args.batch, 3, 224, 224, device="cuda", generator=g).bfloat16().contiguous(memory_format=torch.channels_last)
    inference.calibrate(q, [x[:16].float()])
    q = q.to(memory_format=torch.channels_last)
    q_float = copy.deepcopy(q)                               # the reference's path: TR kernels + cuDNN fp32 conv
    q_tc = copy.deepcopy(q)
    switched, skipped = tr_layer.use_tensor_cores(q_tc)      # every wrapped conv on tcgen05, BN / ReLU / add on torch
    assert len(switched) == 52 and not skipped, skipped
    f = fused.FusedResNet(q)
    paths = {"fused": lambda: f(x),
             "tcgen05": lambda: q_tc(x.float()),
             "float": lambda: q_float(x.float())}
    graphs, outs = {}, {}
    with torch.no_grad():
        for name, fn in paths.items():
            graphs[name], outs[name] = capture(fn)
        for gr in graphs.values():
            gr.replay()
        torch.cuda.synchronize()
        times = {name: [] for name in paths}
        for _ in range(args.rounds):
            for name, gr in graphs.items():
                times[name].append(time_replays(gr, args.replays))
    flop = 2.0 * macs * args.batch
    res = {"what": "ResNet-50 TQ (9-bit, g=8, alpha=12, 3 data terms), random init + randomised BN, bf16 images in HBM, "
                   "CUDA-graph replays alternating per round, TF32 off",
           "gpu": info, "torch": torch.__version__, "batch": args.batch, "rounds": args.rounds, "replays_per_round": args.replays,
           "wrapped_conv_macs_per_image": macs, "paths": {}}
    for name, t in times.items():
        med = statistics.median(t)
        res["paths"][name] = {"ms_median": round(med, 4), "ms_min": round(min(t), 4), "ms_max": round(max(t), 4),
                              "images_per_s": round(args.batch / med * 1e3, 1),
                              "wrapped_conv_tflops": round(flop / (med * 1e-3) / 1e12, 1)}
    scale = float(outs["tcgen05"].abs().max())
    res["fused_vs_tcgen05_logits_rel"] = float((outs["fused"] - outs["tcgen05"]).abs().max()) / scale
    res["fused_vs_float_logits_rel"] = float((outs["fused"] - outs["float"]).abs().max()) / float(outs["float"].abs().max())
    res["speedup_fused_over_tcgen05"] = round(res["paths"]["tcgen05"]["ms_median"] / res["paths"]["fused"]["ms_median"], 3)
    res["speedup_fused_over_float"] = round(res["paths"]["float"]["ms_median"] / res["paths"]["fused"]["ms_median"], 3)
    res["layers"] = layer_plan(f)
    del graphs
    torch.cuda.synchronize()
    try:
        res["eager_fused_split"] = eager_split(f, x)
    except Exception as e:                                   # the timings above stand without it
        res["eager_fused_split"] = {"error": repr(e)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fp:
        json.dump(res, fp, indent=1)
    summary = {k: v for k, v in res.items() if k not in ("layers", "eager_fused_split")}
    print(json.dumps(summary))
    print("engines (engine, groups):", sorted({(l["engine"], l["groups"]) for l in res["layers"]}))


if __name__ == "__main__":
    main()
