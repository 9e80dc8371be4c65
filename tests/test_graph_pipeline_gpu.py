"""The execution path the benchmark times, against eager execution and the CPU emulation.

The other GPU tests call the fused engines eagerly.  `bench.py` times something else: `ShardedInference(cuda_graphs=True)`
captures one forward per input buffer and replays it, `stage()` / `run()` rotate device slots behind a copy stream,
`U8Frontend` feeds uint8 batches through the stem's fold pass, and the gather modes use side streams and rotating
buffers.  What goes wrong there is lifetime and ordering, not rounding: a buffer a captured graph writes that Python has
freed, a slot rewritten before its forward read it, a capture that changes which code runs.  So every result here is
compared bit for bit with eager execution of the same batch (and, where a capture dict exists, with
oracle/fused_emul.py), over several distinct batches, so that a stale or early read shows up as another batch's logits.
"""
import os
import socket
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

pytestmark = pytest.mark.gpu

H, W = 96, 128                      # (H/2) * (W/2) >= 128 with both even: the tensor-core stem runs
CL = torch.channels_last


@pytest.fixture(autouse=True)
def _fp32_math():
    # the float parts (cuDNN stem, classifier) must be true fp32 for the 1e-5 comparisons (TF32 keeps 10 mantissa bits)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _randomise_bn(model, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for mod in model.modules():
            if isinstance(mod, nn.BatchNorm2d):
                n = mod.num_features
                mod.running_mean.copy_(torch.randn(n, device="cuda", generator=g) * 0.2)
                mod.running_var.copy_(torch.rand(n, device="cuda", generator=g) + 0.5)
                mod.weight.copy_(torch.rand(n, device="cuda", generator=g) + 0.5)
                mod.bias.copy_(torch.randn(n, device="cuda", generator=g) * 0.2)


def _tq_model(arch, seed=0):
    """Random-init torchvision model with randomised BatchNorm statistics, TQ-converted at the benchmarked setting
    (9-bit, g=8, alpha=12, 3 data terms), not calibrated yet."""
    import torchvision
    from term_quantization_b200 import cnn_models
    torch.manual_seed(seed)
    base = getattr(torchvision.models, arch)(weights=None).cuda().eval()
    _randomise_bn(base, seed)
    return cnn_models.convert_model(base, cnn_models.static_conv_layer_settings(base, 9, 8, 12), 9, 3)


def _calibrated(arch, calib, seed=0):
    from term_quantization_b200 import inference
    q = _tq_model(arch, seed)
    inference.calibrate(q, [calib])
    return q.to(memory_format=CL)


@pytest.fixture(scope="module")
def resnet():
    calib = torch.randn(4, 3, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    return _calibrated("resnet18", calib)


def _images(kind, n, seed, h=H, w=W):
    """A device batch: bf16 / fp32 [n, 3, h, w] in channels_last memory, or uint8 [n, h, w, 3]."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "uint8":
        return torch.randint(0, 256, (n, h, w, 3), device="cuda", dtype=torch.uint8, generator=g)
    x = torch.randn(n, 3, h, w, device="cuda", generator=g).contiguous(memory_format=CL)
    return x.to(torch.bfloat16 if kind == "bf16" else torch.float32)


def _host(kind, n, seed):
    """The same kinds of batch in pinned host memory, as bench.py stages them (channels_last for the images)."""
    g = torch.Generator().manual_seed(seed)
    if kind == "uint8":
        x = torch.randint(0, 256, (n, H, W, 3), dtype=torch.uint8, generator=g)
        return torch.empty(x.shape, dtype=x.dtype, pin_memory=True).copy_(x)
    dt = torch.bfloat16 if kind == "bf16" else torch.float32
    x = torch.randn(n, 3, H, W, generator=g)
    out = torch.empty(x.shape, dtype=dt, pin_memory=True, memory_format=CL).copy_(x)
    assert out.is_pinned() and out.is_contiguous(memory_format=CL)
    return out


def _front(f, kind):
    from term_quantization_b200 import inference
    return inference.U8Frontend(f) if kind == "uint8" else f


def _all_distinct(logits):
    return all(not torch.equal(logits[i], logits[j]) for i in range(len(logits)) for j in range(i))


def _replay_equals_eager(model, kind, n, h=H, w=W, seeds=(11, 12, 13)):
    """ShardedInference(cuda_graphs=True) on one input buffer; new batches written into it in place; every forward's
    logits against the eager forward of the same batch."""
    from term_quantization_b200 import inference
    batches = [_images(kind, n, s, h, w) for s in seeds]
    with torch.no_grad():
        want = [model(b).clone() for b in batches]
    assert _all_distinct(want)
    runner = inference.ShardedInference(model, "cuda", cuda_graphs=True)
    buf = torch.empty_like(batches[0])
    got = []
    for b in batches:
        buf.copy_(b)
        got.append(runner.forward(buf).clone())
    assert len(runner._graphs) == 1
    for k, (a, b) in enumerate(zip(got, want)):
        assert torch.equal(a, b), f"batch {k}: graph replay differs from eager by {float((a - b).abs().max())}"


# ---- 1. graph replay == eager == emulation, for every executor bench.py / bench_extra.py time ----------------------

@pytest.mark.parametrize("kind", ["bf16", "fp32", "uint8"])
@pytest.mark.parametrize("stem,engine", [("tcgen05", "auto"), ("tcgen05_pool", "auto"), ("cudnn", "auto"), ("tcgen05", "i8")])
def test_resnet_graph_replay_equals_eager(resnet, stem, engine, kind):
    from term_quantization_b200 import fused
    f = fused.FusedResNet(resnet, stem=stem, engine=engine)
    _replay_equals_eager(_front(f, kind), kind, 3)


@pytest.mark.parametrize("kind,n,h,w", [("bf16", 2, 224, 224), ("uint8", 2, 224, 224),
                                        ("bf16", 3, 95, 127), ("uint8", 2, 95, 128)])
def test_resnet_graph_replay_other_shapes(resnet, kind, n, h, w):
    """224^2 (the benchmark's map) and odd maps, which take the cuDNN stem / normalise-first fallback."""
    from term_quantization_b200 import fused
    _replay_equals_eager(_front(fused.FusedResNet(resnet), kind), kind, n, h, w)


def _capture(fn, warmup=2):
    """fn() captured as one CUDA graph the way ShardedInference and bench_extra._time_graphed do it: warm-up on a side
    stream, then capture.  A failing capture raises (no fall-back).  Returns (graph, what fn returned)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warmup):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    return graph, out


def test_resnet_replay_pinned_to_cpu_emulation(resnet):
    """A replay (not only an eager run) against oracle/fused_emul.py: the captured block outputs bit for bit, the logits
    against an fp64 classifier on the emulated features to 1e-5."""
    from oracle import fused_emul
    from term_quantization_b200 import fused
    f = fused.FusedResNet(resnet)
    x = _images("bf16", 2, 20)
    cap = {}
    with torch.no_grad():
        graph, logits = _capture(lambda: f(x, capture=cap))
    desc = f.chain_description()
    fc_w, fc_b = resnet.fc.weight.detach().double().cpu(), resnet.fc.bias.detach().double().cpu()
    seen = []
    for seed in (21, 22):
        x.copy_(_images("bf16", 2, seed))
        graph.replay()
        with torch.no_grad():
            assert torch.equal(logits, f(x))
        seen.append(logits.clone())
        emu = fused_emul.run_resnet_chain(desc, cap["stem"].cpu().numpy())
        got = cap["final"].cpu().numpy()
        assert got.shape == emu.shape
        assert np.array_equal(got.view(np.uint32), emu.view(np.uint32)), \
            f"{int((got != emu).sum())} of {got.size} replayed block outputs differ from the emulation"
        want = torch.from_numpy(emu).double().mean(dim=(1, 2)) @ fc_w.t() + fc_b
        rel = float((logits.double().cpu() - want).abs().max()) / float(want.abs().max())
        assert rel < 1e-5, rel
    assert _all_distinct(seen)


def test_vgg_replay_pinned_to_cpu_emulation():
    from oracle import fused_emul
    from term_quantization_b200 import fused
    x = _images("fp32", 2, 30, 64, 96)
    f = fused.FusedVGG(_calibrated("vgg16_bn", x.clone(), seed=3))
    cap = {}
    with torch.no_grad():
        graph, logits = _capture(lambda: f(x, capture=cap))
    stages = f.chain_description()
    seen = []
    for seed in (31, 32):
        x.copy_(_images("fp32", 2, seed, 64, 96))
        graph.replay()
        with torch.no_grad():
            assert torch.equal(logits, f(x))
        seen.append(logits.clone())
        want = fused_emul.run_vgg_chain(stages, cap["stem_codes"].cpu().numpy().astype(np.int32))
        got = cap["final"].cpu().numpy()
        assert got.shape == want.shape and np.array_equal(got, want), float(np.abs(got - want).max())
    assert _all_distinct(seen)


def test_mobilenet_replay_pinned_to_cpu_emulation():
    from oracle import fused_emul
    from term_quantization_b200 import fused
    x = _images("fp32", 2, 40)
    f = fused.FusedMobileNet(_calibrated("mobilenet_v2", x.clone(), seed=5))
    cap = {}
    with torch.no_grad():
        graph, logits = _capture(lambda: f(x, capture=cap))
    desc = f.chain_description()
    seen = []
    for seed in (41, 42):
        x.copy_(_images("fp32", 2, seed))
        graph.replay()
        with torch.no_grad():
            assert torch.equal(logits, f(x))
        seen.append(logits.clone())
        want = fused_emul.run_mobilenet_chain(desc, cap["stem_codes"].cpu().numpy())
        got = cap["final"].cpu().numpy()
        assert got.shape == want.shape and np.array_equal(got, want), f"{int((got != want).sum())} of {got.size} differ"
    assert _all_distinct(seen)


def test_mlp_on_tensor_cores_captures_and_replays_like_eager():
    """bench_extra's MNIST MLP 784-512-512-10 (wb 4, g=8, alpha=12, db 6) on the tcgen05 linear path, batch 256."""
    from term_quantization_b200 import evaluate_mlp, tr_layer
    from term_quantization_b200.train_mlp import MNISTMLP
    torch.manual_seed(0)
    mlp = MNISTMLP().cuda().eval()
    mlp = evaluate_mlp.replace_linear_layers(mlp, evaluate_mlp.static_linear_layer_settings(mlp, 4, 8, 12), 6, 6)
    g = torch.Generator(device="cuda").manual_seed(50)
    xm = torch.randn(256, 1, 28, 28, device="cuda", generator=g)
    with torch.no_grad():
        mlp(xm)
        tr_layer.set_tr_tracking(mlp, False)
        tr_layer.use_tensor_cores(mlp)
        layers = [m for m in mlp.modules() if isinstance(m, tr_layer.TRLinearLayer)]
        assert len(layers) == 3 and all(m._tc_weight is not None for m in layers)
        graph, out = _capture(lambda: mlp(xm), warmup=3)
        seen = []
        for _ in range(3):
            xm.copy_(torch.randn(256, 1, 28, 28, device="cuda", generator=g))
            graph.replay()
            got = out.clone()
            assert torch.equal(got, mlp(xm))
            seen.append(got)
    assert _all_distinct(seen)


def test_lstm_on_tensor_cores_captures_and_replays_like_eager():
    """TRLSTMLayer 650/650, 2 layers, seq 35 x batch 80 (the Wikitext-2 shape bench_extra times): the integer input
    projection on tcgen05, the step-wise layer 0 and cuDNN's layer 1, captured and replayed."""
    from term_quantization_b200 import tr_layer
    torch.manual_seed(0)
    L = tr_layer.TRLSTMLayer(nn.LSTM(650, 650, 2).cuda().eval(), 8, 8, 8, 8, 12)
    g = torch.Generator(device="cuda").manual_seed(51)
    emb = torch.randn(35, 80, 650, device="cuda", generator=g) * 0.1
    hid = (torch.randn(2, 80, 650, device="cuda", generator=g) * 0.1, torch.randn(2, 80, 650, device="cuda", generator=g) * 0.1)
    with torch.no_grad():
        L(emb, hid)
        tr_layer.set_tr_tracking(L, False)
        L.use_tensor_cores()
        graph, (y, (h, c)) = _capture(lambda: L(emb, hid), warmup=3)
        seen = []
        for _ in range(3):
            emb.copy_(torch.randn(35, 80, 650, device="cuda", generator=g) * 0.1)
            for t in hid:
                t.copy_(torch.randn(2, 80, 650, device="cuda", generator=g) * 0.1)
            graph.replay()
            got = (y.clone(), h.clone(), c.clone())
            ye, (he, ce) = L(emb, hid)
            for a, b in zip(got, (ye, he, ce)):
                assert torch.equal(a, b), float((a - b).abs().max())
            seen.append(got[0])
    assert _all_distinct(seen)


# ---- 2. the staged pipeline (stage ahead, run) == eager, step by step ---------------------------------------------

@pytest.mark.parametrize("kind", ["bf16", "fp32", "uint8"])
@pytest.mark.parametrize("graphs", [True, False])
@pytest.mark.parametrize("slots", [3, 2])
def test_staged_pipeline_equals_eager(resnet, kind, graphs, slots):
    """bench.py's e2e loop: stage `slots - 1` shards ahead (two with the default three slots), then run; ten distinct
    host batches with one change of batch size in the middle (the slots are reallocated; with graphs, the graphs of the
    old buffers keep them)."""
    from term_quantization_b200 import fused, inference
    model = _front(fused.FusedResNet(resnet), kind)
    steps = 10
    host = [_host(kind, 3 if i < steps // 2 else 2, 100 + i) for i in range(steps)]
    with torch.no_grad():
        want = [model(h.cuda()) for h in host]
    assert _all_distinct([w[:2] for w in want])
    runner = inference.ShardedInference(model, "cuda", cuda_graphs=graphs, slots=slots)
    ahead = slots - 1
    staged = [runner.stage(host[i]) for i in range(ahead)]
    got = []
    for i in range(steps):
        if i + ahead < steps:
            staged.append(runner.stage(host[i + ahead]))
        out = runner.run(staged.pop(0))
        got.append(runner._last_local.clone())              # stream-ordered: no synchronise needed
    torch.cuda.current_stream().synchronize()
    assert torch.equal(out, got[-1].cpu())                  # the pinned tensor of the last run()
    if graphs:
        assert len(runner._graphs) == 2 * slots             # one graph per slot buffer and shape, old buffers kept
    for i, (a, b) in enumerate(zip(got, want)):
        assert torch.equal(a, b), f"step {i}: staged logits differ from the eager logits of its batch"


@pytest.mark.parametrize("slots", [3, 2])
def test_staging_more_shards_than_slots_is_refused(resnet, slots):
    """One shard more than there are slots would overwrite a shard that has not run (bench.py's two-ahead loop with two
    slots): refused, not silently run on the wrong batch.  After one run() the freed slot can be staged again."""
    from term_quantization_b200 import fused, inference
    f = fused.FusedResNet(resnet)
    host = [_host("bf16", 2, 120 + i) for i in range(slots + 1)]
    r = inference.ShardedInference(f, "cuda", slots=slots)
    staged = [r.stage(h) for h in host[:slots]]
    with pytest.raises(RuntimeError):
        r.stage(host[slots])
    with torch.no_grad():
        want = f(host[0].cuda())
    r.run(staged[0])
    assert torch.equal(r._last_local, want)
    r.stage(host[slots])


def test_gather_modes_agree_at_world_size_1(resnet):
    """step / async / end give the same logits on one process, and finish() returns None there (nothing outstanding)."""
    from term_quantization_b200 import fused, inference
    f = fused.FusedResNet(resnet)
    batches = [_images("bf16", 2, 60 + k) for k in range(3)]
    with torch.no_grad():
        want = [f(b) for b in batches]
    for gather in ("step", "async", "end"):
        runner = inference.ShardedInference(f, "cuda", cuda_graphs=True, gather=gather)
        buf = torch.empty_like(batches[0])
        for b, w in zip(batches, want):
            buf.copy_(b)
            assert torch.equal(runner.forward(buf), w), gather
        assert runner.finish() is None, gather


# ---- 3. lifetime: every address a live graph writes is owned by that graph or outlives it --------------------------

# scratch-pointer argument of every stem entry point (include/tq_b200.h)
STEM_SCRATCH_ARG = {"tq_stem_conv7x7s2": 1, "tq_stem_conv7x7s2_dt": 2, "tq_stem_conv7x7s2_rowmax": 2,
                    "tq_stem_conv7x7s2_pool_enc": 2, "tq_stem_conv7x7s2_u8": 3, "tq_stem_conv7x7s2_u8_rowmax": 3}


def _record_while_capturing(monkeypatch, args):
    """Wrap library entry points (conv_codes looks them up on every call) to record one pointer argument of every launch
    made under stream capture."""
    from term_quantization_b200 import _lib
    L = _lib.lib()
    seen = []
    for name, k in args.items():
        def wrapped(*a, _fn=getattr(L, name), _k=k, _name=name):
            if torch.cuda.is_current_stream_capturing():
                seen.append((_name, int(a[_k])))
            return _fn(*a)
        monkeypatch.setattr(L, name, wrapped)
    return seen


def _block_of(ptr):
    """(start, requested size, state, pool id) of the caching-allocator block holding device address ptr, or None."""
    for seg in torch.cuda.memory_snapshot():
        if not seg["address"] <= ptr < seg["address"] + seg["total_size"]:
            continue
        start = seg["address"]
        for b in seg["blocks"]:
            start = b.get("address", start)
            if start <= ptr < start + b["size"]:
                return start, b.get("requested_size"), b["state"], tuple(seg.get("segment_pool_id", ()))
            start += b["size"]
    return None


def _still_owned(graph, ptr, at_capture):
    """In the graph's private pool, or the very allocation (same start and size, still active) it was at capture."""
    now = _block_of(ptr)
    if now is None:
        return False
    if graph is not None and now[3] == tuple(graph.pool()):
        return True
    return now[2] == "active_allocated" and at_capture is not None and now[:2] == at_capture[:2]


def test_captured_stems_write_only_owned_memory(resnet, monkeypatch):
    """One FusedResNet, two executors: graph A (bf16, batch 2), then graph B (fp32, batch 4: a larger folded image),
    then a uint8 graph (batch 2).  Before any further replay, every scratch address the captured stem kernels write must
    still be owned; then replays with new contents equal eager."""
    from term_quantization_b200 import fused, inference
    f = fused.FusedResNet(resnet)
    seen = _record_while_capturing(monkeypatch, STEM_SCRATCH_ARG)
    r16 = inference.ShardedInference(f, "cuda", cuda_graphs=True)
    r8 = inference.ShardedInference(inference.U8Frontend(f), "cuda", cuda_graphs=True)
    live = []
    for name, runner, kind, n in (("A bf16 x2", r16, "bf16", 2), ("B fp32 x4", r16, "fp32", 4), ("uint8 x2", r8, "uint8", 2)):
        buf = _images(kind, n, 70)
        n0 = len(seen)
        runner.forward(buf)                                  # warm-up, capture, first replay
        graph = runner._graphs[(buf.data_ptr(), tuple(buf.shape), tuple(buf.stride()), buf.dtype)][0]
        ptrs = [p for _, p in seen[n0:]]
        assert ptrs, f"{name}: no stem launch recorded while capturing"
        live.append((name, runner, kind, buf, graph, [(p, _block_of(p)) for p in ptrs]))
    for name, _, _, _, graph, recs in live:
        for p, then in recs:
            assert _still_owned(graph, p, then), \
                f"graph {name}: its stem writes {p:#x}, which it no longer owns (block now {_block_of(p)}, at capture {then})"
    for name, runner, kind, buf, _, _ in live:
        for seed in (71, 72):
            buf.copy_(_images(kind, buf.shape[0], seed))
            got = runner.forward(buf).clone()
            with torch.no_grad():
                assert torch.equal(got, runner.model(buf)), name


def test_captured_raw_i8_conv_keeps_its_weight_planes(monkeypatch):
    """conv2d_codes(engine='i8') without plan= is captured, then more than 256 other weights go through the raw op.  The
    int8 weight planes the graph reads must still be owned, and a replay must equal eager and the exact integer conv."""
    from term_quantization_b200 import conv_codes
    g = torch.Generator(device="cuda").manual_seed(80)
    act = torch.randint(0, 257, (2, 12, 20, 32), device="cuda", generator=g).half()
    wgt = torch.randint(-100, 101, (9, 64, 32), device="cuda", generator=g).half()
    seen = _record_while_capturing(monkeypatch, {"tq_conv2d_planes_i8_enc": 1})

    def conv():
        return conv_codes.conv2d_codes(act, wgt, None, (3, 3), 1, 1, 1.0, engine="i8")
    graph, out = _capture(conv)
    recs = [(p, _block_of(p)) for _, p in seen]
    assert recs, "no i8 conv launch recorded while capturing"
    small = torch.randint(0, 9, (1, 4, 4, 16), device="cuda", generator=g).half()
    others = [torch.randint(-8, 9, (1, 16, 16), device="cuda", generator=g).half() for _ in range(300)]
    for w in others:
        conv_codes.conv2d_codes(small, w, None, (1, 1), 1, 0, 1.0, engine="i8")
    for p, then in recs:
        assert _still_owned(None, p, then), \
            f"the captured i8 conv reads weight planes at {p:#x}, no longer owned (block now {_block_of(p)}, at capture {then})"
    act.copy_(torch.randint(0, 257, act.shape, device="cuda", generator=g).half())
    graph.replay()
    assert torch.equal(out, conv())
    w4 = wgt.double().view(3, 3, 64, 32).permute(2, 3, 0, 1)
    exact = torch.nn.functional.conv2d(act.double().permute(0, 3, 1, 2), w4, None, 1, 1).permute(0, 2, 3, 1)
    assert torch.equal(out.double(), exact)


# ---- 4. two ranks over NCCL ----------------------------------------------------------------------------------------

def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from term_quantization_b200 import fused, inference, tr_layer
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        n = 4
        g = torch.Generator(device=dev).manual_seed(90)          # the whole job's batches, the same on every rank
        batches = [torch.randn(n, 3, H, W, device=dev, generator=g).bfloat16().contiguous(memory_format=CL) for _ in range(3)]
        bounds = [inference.shard_bounds(n, world, r) for r in range(world)]
        lo, hi = bounds[rank]
        q = _tq_model("resnet18")
        inference.calibrate(q, [batches[0][lo:hi].float()])     # this rank's shard, histograms summed over ranks
        ref = _tq_model("resnet18")                             # one process calibrating on the whole batch
        tr_layer.set_tr_tracking(ref, True)
        with torch.no_grad():
            ref(batches[0].float())
        tr_layer.set_tr_tracking(ref, False)
        sfs = [m.input_quant.sf for m in q.modules() if isinstance(m, tr_layer.TRConv2dLayer)]
        sfs_ref = [m.input_quant.sf for m in ref.modules() if isinstance(m, tr_layer.TRConv2dLayer)]
        res = {"sf": len(sfs) == 19 and sfs == sfs_ref}
        f = fused.FusedResNet(q.to(memory_format=CL))
        with torch.no_grad():
            # rank-major: shard 0's logits, then shard 1's (each shard's eager forward), and the whole batch at once
            want = [torch.cat([f(b[a:z]) for a, z in bounds]) for b in batches]
            whole = [f(b) for b in batches]
        res["whole"] = all(float((w - v).abs().max()) <= 1e-5 * float(v.abs().max()) for w, v in zip(want, whole))
        for gather in ("step", "async", "end"):
            runner = inference.ShardedInference(f, dev, cuda_graphs=True, gather=gather)
            buf = torch.empty_like(batches[0][lo:hi])
            got = []
            for b in batches:
                buf.copy_(b[lo:hi])
                out = runner.forward(buf)
                if gather == "step":
                    got.append(out.clone())
                elif gather == "async":
                    got.append(runner.finish().clone())        # completes this step's gather
            if gather == "end":
                fin = runner.finish()
                got = list(fin) if fin is not None and tuple(fin.shape) == (3, n, 1000) else []
            else:
                assert runner.finish() is None or gather == "async"
            res[gather] = len(got) == 3 and all(torch.equal(a, b) for a, b in zip(got, want))
        ret[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two visible GPUs")
def test_two_ranks_over_nccl():
    """Calibration on shards with summed histograms gives the whole batch's scale factors, and the graph-replayed
    forward gathers every rank's logits rank-major in all three gather modes."""
    world = 2
    port = _free_port()
    with mp.Manager() as mgr:
        ret = mgr.dict()
        ctx = mp.spawn(_nccl_worker, args=(world, port, ret), nprocs=world, join=False)
        deadline = time.monotonic() + 900
        try:
            while not ctx.join(timeout=5):
                assert time.monotonic() < deadline, "the ranks did not finish in 15 minutes"
        finally:
            for p in ctx.processes:
                if p.is_alive():
                    p.terminate()
            for p in ctx.processes:
                p.join(30)
        want = {"sf": True, "whole": True, "step": True, "async": True, "end": True}
        assert dict(ret) == {0: want, 1: want}
