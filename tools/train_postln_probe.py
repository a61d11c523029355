#!/usr/bin/env python
"""Post-LN against pre-LN training step at the BASELINE config-5 shape (Large, 8 clips x 150 frames, bf16, loss =
mean(y^2), forward + backward, no regularisation, no all-reduce).  Both orders run the same GEMMs and 2L + 1 LayerNorms;
this measures what the different LayerNorm backward and the extra saved activations cost.  Orders alternated in one
process, each window timed with CUDA events on a non-default stream (the library replays its launch lists as CUDA
graphs there).
  tail     AVHubertModel.extract_finetune with frozen feature extractors (feature_grad_mult = 0; the frozen extractors'
           forward is part of the step)
  encoder  the bare TransformerEncoder(args, trainable=True) on [8, 150, 1024]
  python tools/train_postln_probe.py [--rounds R] [--steps K] [--out profiles/train_postln_probe.json]      (needs a B200)"""
import argparse
import json
import os
import subprocess
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5, help="steps per timed window")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "train_postln_probe.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    from multimodalvc_b200 import AVHubertConfig, AVHubertModel, _lib
    from multimodalvc_b200.sr_predictor import TransformerEncoder
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(500)
    v = torch.randn(8, 1, 150, 88, 88, generator=g).to(dev, torch.bfloat16)
    a = torch.randn(8, 104, 150, generator=g).to(dev, torch.bfloat16)
    x = torch.randn(8, 150, 1024, generator=g).to(dev, torch.bfloat16)
    np.random.seed(0)
    torch.manual_seed(0)
    result = {"card": card(), "shape": "large, 8 x 150, bf16", "rounds": args.rounds, "steps_per_window": args.steps}
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))

    def tail_step(lnf):
        m = AVHubertModel(AVHubertConfig.named("large", feature_grad_mult=0.0, trainable=True, layer_norm_first=lnf,
                                               attention_dropout=0.0, dropout_input=0.0, dropout=0.0,
                                               activation_dropout=0.0, encoder_layerdrop=0.0))
        m.remove_pretraining_modules()
        m = m.to(dev, torch.bfloat16).train()
        params = m.tail_parameters()

        def step():
            y, _ = m.extract_finetune({"audio": a, "video": v}, None)
            y.float().pow(2).mean().backward()
            for p in params:
                p.grad = None
        return m, step

    def encoder_step(lnf):
        enc = TransformerEncoder(SimpleNamespace(
            encoder_embed_dim=1024, encoder_ffn_embed_dim=4096, encoder_attention_heads=16, encoder_layers=24,
            conv_pos=128, conv_pos_groups=16, layer_norm_first=lnf, activation_fn="gelu", dropout=0.0,
            attention_dropout=0.0, activation_dropout=0.0, encoder_layerdrop=0.0), trainable=True)
        enc = enc.to(dev, torch.bfloat16).train()

        def step():
            xd = x.detach().requires_grad_(True)
            y, _ = enc(xd)
            y.float().pow(2).mean().backward()
            for p in enc.parameters():
                p.grad = None
        return enc, step

    for kind, make in (("tail", tail_step), ("encoder", encoder_step)):
        orders = {"pre_ln": True, "post_ln": False}
        steps, mods, launches = {}, {}, {}
        times = {k: [] for k in orders}
        with torch.cuda.stream(stream):
            for name, lnf in orders.items():      # warm-up: first run, graph capture, replay
                mods[name], steps[name] = make(lnf)
                for _ in range(3):
                    steps[name]()
                torch.cuda.synchronize(dev)
                _lib.reset_launch_count()
                steps[name]()
                torch.cuda.synchronize(dev)
                launches[name] = _lib.launch_count()
            for _ in range(args.rounds):
                for name in orders:
                    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    t0.record()
                    for _ in range(args.steps):
                        steps[name]()
                    t1.record()
                    torch.cuda.synchronize(dev)
                    times[name].append(t0.elapsed_time(t1) / args.steps)
        med = {k: float(np.median(t)) for k, t in times.items()}
        result[kind] = {"ms_per_step_median": med, "ms_per_step_all": times, "launches_per_step": launches,
                        "post_vs_pre_pct": 100.0 * (med["post_ln"] / med["pre_ln"] - 1.0)}
        del mods, steps
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if "all" not in kk})
                      for k, v in result.items()}, indent=1))


if __name__ == "__main__":
    main()
