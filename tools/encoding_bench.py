"""Throughput of the fused ResNet-18 engine per term encoding (HESE, binary, Booth).

Same workload as bench.py's headline (batch 256 of 224x224 bf16 images, 9-bit weights, g = 8, alpha = 12, 9-bit data with
3 terms, fused.FusedResNet replayed as one CUDA graph per forward by inference.ShardedInference), with every wrapped
conv converted under the given encoding.  Prints one JSON line per encoding: images/s and engines_per_layer, the
engine the static exactness proof picked for each of the 19 wrapped convs ('f16 xG' = kind::f16 with G K-chunk
accumulators, 'i8 Pw-plane' = kind::i8 planes).  Booth weight codes reach 2^bits where HESE's stop at 2^(bits-1), so
its proofs may need more K chunks or the i8 engine.

    python tools/encoding_bench.py [--steps 30] [--warmup 5] [--batch 256] [--encodings hese binary booth]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def engines_per_layer(f):
    out = []
    for blk in f.blocks:
        for c in blk:
            if c is not None:
                out.append(f"f16 x{c.plan.groups}" if c.plan.engine == "f16" else f"i8 {c.plan.planes_w}w-plane")
    return out


def run(encoding, batch, steps, warmup):
    from torchvision.models import resnet18
    from term_quantization_b200 import cnn_models, fused, inference
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = resnet18(weights=None).eval().to(dev)
    params = cnn_models.static_conv_layer_settings(model, 9, 8, 12)
    q = cnn_models.convert_model(model, params, 9, 3, encoding=encoding).eval()
    gen = torch.Generator(device=dev).manual_seed(0)
    images = [torch.randn(batch, 3, 224, 224, device=dev, generator=gen).bfloat16().float() for _ in range(2)]
    inference.calibrate(q, [images[0][:64]])
    q = q.to(memory_format=torch.channels_last)
    f = fused.FusedResNet(q)
    images = [im.contiguous(memory_format=torch.channels_last).bfloat16() for im in images]
    runner = inference.ShardedInference(f, dev, cuda_graphs=True)
    for i in range(warmup):
        runner.forward(images[i % 2])
    runner.finish()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        runner.forward(images[i % 2])
    runner.finish()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    eng = engines_per_layer(f)
    return {"encoding": encoding, "batch": batch, "steps": steps, "images_per_s": batch * steps / (ms / 1e3),
            "ms_per_step": ms / steps, "engines_per_layer": eng,
            "engine_counts": {k: eng.count(k) for k in sorted(set(eng))}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--encodings", nargs="+", default=["hese", "binary", "booth"], choices=["hese", "binary", "booth"])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("encoding_bench measures the fused engine on a GPU: no CUDA device")
    print(json.dumps(gpu_info()), flush=True)
    for enc in args.encodings:
        print(json.dumps(run(enc, args.batch, args.steps, args.warmup)), flush=True)


if __name__ == "__main__":
    main()
