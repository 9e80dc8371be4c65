"""The Wikitext-2 LSTM workload of bench_extra.py (configs[4]: 650/650, 2 layers, vocab 33,278, seq 35 x batch 80; TQ wb 8,
g 8, alpha 12, db 8, seed 0) on its three paths, timed as CUDA-graph replays in one process, alternating:

  strict   the reference forward as shipped: cuDNN LSTM on quantised emb / h0 / c0, fp32 decoder on the raw input
  tcgen05  tr_layer.use_tensor_cores: layer-0 input projection and decoder on term codes, step-wise layer 0, cuDNN layer 1
  fused    fused.FusedLSTM: the same contractions, every layer's recurrence one persistent kernel (tq_lstm_recurrence)

Then a separate eager pass splits the fused forward into phases with CUDA events, and the recurrence kernel's FFMA rate
is set against a DERIVED fp32 rate (SMs x 128 FMA/clk x the max SM clock nvidia-smi reports; not a measured peak).
Writes DIR/lstm_bench.json.  Usage: python tools/lstm_bench.py --out DIR [--rounds 15] [--replays 20]

--nll times the fused perplexity step instead, as alternating CUDA-graph replays of
  forward + nll_loss                FusedLSTM.forward (log_softmax over the vocabulary) and nll_loss(reduction='none')
  decoder output + log_softmax_nll  the chain up to the padded decoder output, then one tq_log_softmax_nll pass over it
  nll                               FusedLSTM.nll: the decoder's loss epilogue, no [T*B, V] tensor written at all
with the peak memory of each, plus the decoder with its loss epilogue against the decoder followed by
tq_log_softmax_nll (CUDA events over many calls).  Writes DIR/lstm_nll_epilogue.json.

--model GRU RNN_TANH RNN_RELU times the same workload with each of those cells (only the decoder is a TR layer, as in
the reference), one perplexity step as alternating CUDA-graph replays of
  tcgen05  cuDNN recurrence + the decoder on term codes + log_softmax + nll_loss(reduction='none')
  nll      FusedRNN.nll: the recurrence kernel per layer, the decoder's loss epilogue
with the peak memory of each, and every layer's recurrence launch on its own (CUDA events) with its FFMA rate against
the derived fp32 rate.  Writes DIR/rnn_bench.json."""
import argparse
import copy
import gc
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from term_quantization_b200 import conv_codes, evaluate_lstm, fused, tr_cuda, tr_layer  # noqa: E402
from term_quantization_b200.lstm_models.model import RNNModel  # noqa: E402

T, B, H = 35, 80, 650


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                              capture_output=True, text=True, check=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = (v.strip() for v in line.split(","))
        return {"name": name, "power_limit_w": float(power), "max_sm_clock_mhz": float(clock)}
    except Exception as e:                                   # reported, never guessed
        return {"error": f"nvidia-smi query failed: {e}"}


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


def phases(f, tokens, hidden, reps):
    """Eager fused forward split by CUDA events: the same calls FusedLSTM.forward makes, one event between phases."""
    model = f.model
    rnn, dec = model.rnn, model.decoder
    names = []
    times = {}

    def run():
        ev = [torch.cuda.Event(enable_timing=True)]
        ev[0].record()
        labels = []

        def mark(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            ev.append(e)
            labels.append(name)
        emb = model.encoder(tokens)
        h0, c0 = (rnn.input_quant(h) for h in hidden)
        mark("embedding + h0/c0 quantiser")
        y = None
        for l, (w_ih, w_hh, bias) in enumerate(f.layers):
            if l == 0:
                gin = rnn.input_projection(emb)
                mark("layer 0 input projection (tcgen05, term codes)")
            else:
                gin = torch.mm(y.view(T * B, -1), w_ih.t()).view(T, B, -1)
                mark(f"layer {l} input GEMM (fp32)")
            y, _, _ = conv_codes.lstm_recurrence(gin, bias, w_hh, h0[l].contiguous(), c0[l].contiguous())
            mark(f"layer {l} recurrence (tq_lstm_recurrence)")
        q = dec.input_quant
        codes = torch.zeros((T * B, dec._tc_weight.shape[2]), dtype=torch.float16, device=y.device)
        codes[:, :H] = tr_cuda.tr_codes(y.view(1, -1, 1, 1), q.sf, q.data_bits, 1, q.data_terms, dtype=torch.float16,
                                        encoding=q.encoding).view(T * B, H)
        decoded = conv_codes.linear_codes(codes, dec._tc_weight, f.dec_scale, bias=f.dec_bias,
                                          out_features=dec.linear.out_features, plan=dec._tc_plan)
        mark("decoder: encode + linear on term codes (tcgen05)")
        torch.log_softmax(decoded, dim=1)
        mark("log_softmax")
        torch.cuda.synchronize()
        return labels, [ev[i].elapsed_time(ev[i + 1]) for i in range(len(labels))]

    with torch.no_grad():
        for _ in range(3):
            run()
        for _ in range(reps):
            labels, ms = run()
            names = labels
            for k, v in zip(labels, ms):
                times.setdefault(k, []).append(v)
    return [{"phase": k, "ms_median": statistics.median(times[k]), "ms_best": min(times[k])} for k in names]


def _events(fn, launches, samples):
    """Median and best ms per call of fn over `samples` windows of `launches` back-to-back calls (CUDA events)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        fn()
    acc = []
    for _ in range(samples):
        e0.record()
        for _ in range(launches):
            fn()
        e1.record()
        torch.cuda.synchronize()
        acc.append(e0.elapsed_time(e1) / launches)
    return {"ms_median": statistics.median(acc), "ms_best": min(acc), "ms_spread": max(acc) - min(acc)}


def peak_rise(fn):
    """Bytes the caching allocator's peak rises above what is allocated before an eager call of fn."""
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - base
    del out
    return rise


def nll_bench(f, tokens, hidden, targets, rounds, replays, launches=50, samples=10):
    """The fused perplexity step three ways, and the decoder with its loss epilogue against the decoder + one-pass loss."""
    dec = f.model.decoder
    V = dec.linear.out_features
    paths = {"forward + nll_loss": lambda: F.nll_loss(f(tokens, hidden)[0], targets, reduction="none"),
             "decoder output + log_softmax_nll": lambda: conv_codes.log_softmax_nll(f._decoded(tokens, hidden)[0], targets),
             "nll": lambda: f.nll(tokens, targets, hidden)[0]}
    graphs, outs = {}, {}
    for name, fn in paths.items():
        graphs[name], outs[name] = capture(fn)
    samples_ms = {k: [] for k in graphs}
    for _ in range(rounds):
        for name, g in graphs.items():
            samples_ms[name].append(time_replays(g, replays))
    ref = outs["forward + nll_loss"].double()
    rel = {k: float(((outs[k].double() - ref).abs() / ref.abs().clamp(min=1.0)).max()) for k in outs}
    peaks = {k: peak_rise(fn) for k, fn in paths.items()}

    codes = f._decoder_codes(tokens, hidden)[0]              # the decoder's fp16 input codes [T*B, Kp]
    plan, w, scale, bias = dec._tc_plan, dec._tc_weight, f.dec_scale, f.dec_bias
    kernels = {
        "decoder + loss epilogue (linear_codes_nll)":
            lambda: conv_codes.linear_codes_nll(codes, w, scale, targets, bias=bias, out_features=V, plan=plan),
        "decoder (linear_codes) + tq_log_softmax_nll":
            lambda: conv_codes.log_softmax_nll(conv_codes.linear_codes(codes, w, scale, bias=bias, out_features=V,
                                                                       plan=plan), targets),
        "decoder alone (linear_codes)": lambda: conv_codes.linear_codes(codes, w, scale, bias=bias, out_features=V,
                                                                        plan=plan),
    }
    k_times = {}
    for _ in range(2):                                        # alternating, twice: the spread between windows is reported
        for k, fn in kernels.items():
            k_times.setdefault(k, []).append(_events(fn, launches, samples))
    k_res = {k: {"ms_median": statistics.median(r["ms_median"] for r in v), "ms_best": min(r["ms_best"] for r in v),
                 "ms_spread": max(max(r["ms_median"] for r in v) - min(r["ms_median"] for r in v),
                                  max(r["ms_spread"] for r in v))} for k, v in k_times.items()}
    steps = {k: {"ms_best": min(v), "ms_median": statistics.median(v), "ms_spread": max(v) - min(v),
                 "tokens_per_s_median": T * B / statistics.median(v) * 1e3,
                 "peak_memory_rise_bytes": peaks[k], "loss_max_rel_diff_vs_forward_nll_loss": rel[k]}
             for k, v in samples_ms.items()}
    r05, new = steps["decoder output + log_softmax_nll"]["ms_median"], steps["nll"]["ms_median"]
    return {
        "timed_as": f"CUDA-graph replays of the whole step, {replays} per sample, {rounds} rounds alternating the three "
                    "paths; TF32 off.  Peak memory: eager call, rise of max_memory_allocated above the allocation before it",
        "paths": steps,
        "nll_vs_r05_path_ms_saved_median": r05 - new,
        "nll_vs_r05_path_speedup_median": r05 / new,
        "logits_bytes": T * B * V * 4,
        "decoder_kernels": {
            "how": f"eager, CUDA events around {launches} back-to-back calls, {samples} samples, two alternating passes; "
                   f"{T * B} x {V} logits from K = {codes.shape[1]} codes on the '{plan.engine}' engine "
                   f"({plan.groups} K chunk(s)); ms_spread: the widest gap between samples or passes",
            **k_res,
        },
    }


def derived_fp32_rate(info, props):
    """SMs x 128 FP32 FMA/clk x the max SM clock nvidia-smi reports (derived, not a measured peak); None without it."""
    return props.multi_processor_count * 128 * info["max_sm_clock_mhz"] * 1e6 if "max_sm_clock_mhz" in info else None


def rnn_bench(cell, dev, rounds, replays, derived, launches=20, samples=10):
    """One cell's perplexity step on both paths, and its recurrence launches alone."""
    torch.manual_seed(0)
    gen = torch.Generator(device=dev).manual_seed(0)
    base = RNNModel(cell, evaluate_lstm.NTOKENS, 650, 650, 2, 0.5, True).to(dev).eval()
    q = evaluate_lstm.convert_model(base, evaluate_lstm.static_lstm_layer_settings(base, 8, 8, 12), 8, 8)
    tokens = torch.randint(evaluate_lstm.NTOKENS, (T, B), device=dev, generator=gen)
    targets = torch.randint(evaluate_lstm.NTOKENS, (T * B,), device=dev, generator=gen)
    hidden = base.init_hidden(B)
    with torch.no_grad():
        q(tokens, hidden)
        tr_layer.set_tr_tracking(q, False)
        q_tc = copy.deepcopy(q)
        tr_layer.use_tensor_cores(q_tc)
        f = fused.FusedRNN(copy.deepcopy(q))
        paths = {"tcgen05": lambda: F.nll_loss(q_tc(tokens, hidden)[0], targets, reduction="none"),
                 "nll": lambda: f.nll(tokens, targets, hidden)[0]}
        graphs, outs = {}, {}
        for name, fn in paths.items():
            graphs[name], outs[name] = capture(fn)
        samples_ms = {k: [] for k in graphs}
        for _ in range(rounds):
            for name, g in graphs.items():
                samples_ms[name].append(time_replays(g, replays))
        ref = outs["tcgen05"].double()
        rel = float(((outs["nll"].double() - ref).abs() / ref.abs().clamp(min=1.0)).max())
        peaks = {k: peak_rise(fn) for k, fn in paths.items()}

        # every layer's recurrence alone, on the input projection the executor computes for it
        G = conv_codes.RECURRENCE_GATES[cell]
        fma = T * B * G * H * H
        y = f.model.encoder(tokens)
        recurrence = []
        for l, (w_ih, b_gemm, w_hh, b_rec) in enumerate(f.layers):
            x = y.view(T * B, -1)
            gin = (torch.mm(x, w_ih.t()) if b_gemm is None else torch.addmm(b_gemm, x, w_ih.t())).view(T, B, -1)
            h0 = hidden[l].contiguous()
            if cell == "GRU":
                run = lambda gin=gin, b=b_rec, w=w_hh, h0=h0: conv_codes.gru_recurrence(gin, b, w, h0)  # noqa: E731
            else:
                run = lambda gin=gin, b=b_rec, w=w_hh, h0=h0: conv_codes.rnn_recurrence(  # noqa: E731
                    gin, b, w, h0, f.nonlinearity)
            t = _events(run, launches, samples)
            rate = fma / (t["ms_median"] * 1e-3)
            recurrence.append({"layer": l, "fma": fma, **t, "fma_per_s": rate, "fp32_tflops": 2 * rate / 1e12,
                               "share_of_derived_fp32_rate": rate / derived if derived else None})
            y = run()[0]
    steps = {k: {"ms_best": min(v), "ms_median": statistics.median(v), "ms_spread": max(v) - min(v),
                 "tokens_per_s_median": T * B / statistics.median(v) * 1e3, "peak_memory_rise_bytes": peaks[k]}
             for k, v in samples_ms.items()}
    return {"paths": steps, "nll_vs_tcgen05_speedup_median": steps["tcgen05"]["ms_median"] / steps["nll"]["ms_median"],
            "loss_max_rel_diff_nll_vs_tcgen05": rel, "max_hidden": conv_codes.recurrence_max_hidden(cell, dev),
            "recurrence_kernel": {"how": f"eager, CUDA events around {launches} back-to-back launches, {samples} samples",
                                  "layers": recurrence}}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="output directory (lstm_bench.json)")
    ap.add_argument("--rounds", type=int, default=15, help="alternating rounds; each times every path once")
    ap.add_argument("--replays", type=int, default=20, help="graph replays per timed sample")
    ap.add_argument("--nll", action="store_true", help="time the three perplexity paths (lstm_nll_epilogue.json)")
    ap.add_argument("--model", nargs="+", choices=["GRU", "RNN_TANH", "RNN_RELU"],
                    help="time these cells' perplexity step instead (rnn_bench.json)")
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("lstm_bench needs a CUDA device: nothing is timed on the CPU")
    os.makedirs(args.out, exist_ok=True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda")
    info = gpu_info()
    props = torch.cuda.get_device_properties(dev)
    if args.model:
        derived = derived_fp32_rate(info, props)
        res = {"workload": "Wikitext-2-shaped RNNModel 650/650 tied, 2 layers, vocab 33,278, seq 35 x batch 80, only the "
                           "decoder TQ (wb 8 / g 8 / alpha 12 / db 8), seed 0: one perplexity step",
               "gpu": info, "sms": props.multi_processor_count,
               "timed_as": f"CUDA-graph replays of the whole step, {args.replays} per sample, {args.rounds} rounds "
                           "alternating the two paths; TF32 off.  Peak memory: eager call, rise of max_memory_allocated "
                           "above the allocation before it",
               "derived_fp32_fma_rate": {"fma_per_s": derived, "how": "SMs x 128 FP32 FMA/clk x max SM clock (derived, "
                                                                      "not a measured peak)"},
               "cells": {cell: rnn_bench(cell, dev, args.rounds, args.replays, derived) for cell in args.model}}
        path = os.path.join(args.out, "rnn_bench.json")
        with open(path, "w") as fp:
            json.dump(res, fp, indent=1)
        print(json.dumps(res, indent=1))
        return

    torch.manual_seed(0)
    gen = torch.Generator(device=dev).manual_seed(0)
    base = RNNModel('LSTM', evaluate_lstm.NTOKENS, 650, 650, 2, 0.5, True).to(dev).eval()
    q = evaluate_lstm.convert_model(base, evaluate_lstm.static_lstm_layer_settings(base, 8, 8, 12), 8, 8)
    tokens = torch.randint(evaluate_lstm.NTOKENS, (T, B), device=dev, generator=gen)
    hidden = base.init_hidden(B)
    with torch.no_grad():
        q(tokens, hidden)
        tr_layer.set_tr_tracking(q, False)
        q_tc = copy.deepcopy(q)
        tr_layer.use_tensor_cores(q_tc)
        f = fused.FusedLSTM(copy.deepcopy(q))
        if args.nll:
            targets = torch.randint(evaluate_lstm.NTOKENS, (T * B,), device=dev, generator=gen)
            res = {"workload": "Wikitext-2-shaped LSTM 650/650 tied, 2 layers, vocab 33,278, seq 35 x batch 80, TQ wb 8 / "
                               "g 8 / alpha 12 / db 8 (bench_extra.py configs[4]), seed 0: one perplexity step",
                   "gpu": info, "sms": props.multi_processor_count,
                   **nll_bench(f, tokens, hidden, targets, args.rounds, args.replays)}
            path = os.path.join(args.out, "lstm_nll_epilogue.json")
            with open(path, "w") as fp:
                json.dump(res, fp, indent=1)
            print(json.dumps(res, indent=1))
            return
        paths = {"strict": lambda: q(tokens, hidden), "tcgen05": lambda: q_tc(tokens, hidden),
                 "fused": lambda: f(tokens, hidden)}
        graphs, outs, errors = {}, {}, {}
        for name, fn in paths.items():
            try:
                graphs[name], outs[name] = capture(fn)
            except Exception as e:                           # a refused capture is a result: report it
                errors[name] = f"{type(e).__name__}: {e}"
        samples = {k: [] for k in graphs}
        for _ in range(args.rounds):
            for name, g in graphs.items():
                samples[name].append(time_replays(g, args.replays))
        check = {}
        if "fused" in outs and "tcgen05" in outs:
            (lf, (hf, cf)), (lt, (ht, ct)) = outs["fused"], outs["tcgen05"]
            check = {"hn_max_abs_diff": float((hf - ht).abs().max()), "cn_max_abs_diff": float((cf - ct).abs().max()),
                     "log_probs_mean_abs_diff": float((lf - lt).abs().mean())}
    per_phase = phases(f, tokens, hidden, reps=20)
    rec = [p for p in per_phase if "recurrence" in p["phase"]]
    fma = T * B * 4 * H * H
    derived = derived_fp32_rate(info, props)
    recurrence = []
    for p in rec:
        rate = fma / (p["ms_median"] * 1e-3)
        recurrence.append({"phase": p["phase"], "fma": fma, "ms_median": p["ms_median"], "fma_per_s": rate,
                           "fp32_tflops": 2 * rate / 1e12,
                           "share_of_derived_fp32_rate": rate / derived if derived else None})
    res = {
        "workload": "Wikitext-2-shaped LSTM 650/650 tied, 2 layers, vocab 33,278, seq 35 x batch 80, TQ wb 8 / g 8 / "
                    "alpha 12 / db 8 (bench_extra.py configs[4]), seed 0",
        "gpu": info, "sms": props.multi_processor_count, "shared_memory_per_block_optin": props.shared_memory_per_block_optin,
        "lstm_max_hidden": conv_codes.lstm_max_hidden(dev),
        "timed_as": f"CUDA-graph replays, {args.replays} per sample, {args.rounds} rounds alternating the paths; "
                    "TF32 off",
        "paths": {k: {"ms_best": min(v), "ms_median": statistics.median(v),
                      "tokens_per_s_median": T * B / statistics.median(v) * 1e3} for k, v in samples.items()},
        "capture_errors": errors,
        "fused_vs_tcgen05": check,
        "fused_phases_eager": per_phase,
        "recurrence_kernel": recurrence,
        "derived_fp32_fma_rate": {"fma_per_s": derived, "how": "SMs x 128 FP32 FMA/clk x max SM clock (derived, "
                                                                "not a measured peak)"},
    }
    path = os.path.join(args.out, "lstm_bench.json")
    with open(path, "w") as fp:
        json.dump(res, fp, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
