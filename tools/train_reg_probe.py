#!/usr/bin/env python
"""Cost of dropout / LayerDrop in the fine-tuning step (BASELINE config 5 shape: Large, 8 clips x 150 frames, bf16,
loss = mean(y^2), forward + backward, no all-reduce): settings alternated in one process, each timed with CUDA events on
a non-default stream (the library replays its launch lists as CUDA graphs there).
  off        every regulariser 0 (the plain plan: what bench.py config 5 runs)
  dropout    dropout = activation_dropout = dropout_input = 0.1, no LayerDrop
  ld_keep    the same + a LayerDrop plan whose coins drop nothing (encoder_layerdrop 1e-12)
  ld_0.1     the same with encoder_layerdrop 0.1 and real coins (a step runs ~90 % of the layers)
  python tools/train_reg_probe.py [--rounds R] [--steps K] [--out profiles/train_reg_probe.json]      (needs a B200)"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SETTINGS = {
    "off": dict(dropout_input=0.0, dropout=0.0, activation_dropout=0.0, encoder_layerdrop=0.0),
    "dropout": dict(dropout_input=0.1, dropout=0.1, activation_dropout=0.1, encoder_layerdrop=0.0),
    "ld_keep": dict(dropout_input=0.1, dropout=0.1, activation_dropout=0.1, encoder_layerdrop=1e-12),
    "ld_0.1": dict(dropout_input=0.1, dropout=0.1, activation_dropout=0.1, encoder_layerdrop=0.1),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5, help="steps per timed window")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "train_reg_probe.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    from multimodalvc_b200 import AVHubertConfig, AVHubertModel, _lib
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(500)
    v = torch.randn(8, 1, 150, 88, 88, generator=g).to(dev, torch.bfloat16)
    a = torch.randn(8, 104, 150, generator=g).to(dev, torch.bfloat16)
    np.random.seed(0)
    torch.manual_seed(0)
    result = {"card": card(), "shape": "large, 8 x 150, bf16", "rounds": args.rounds, "steps_per_window": args.steps}
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    for fgm in (0.1, 0.0):
        m = AVHubertModel(AVHubertConfig.named("large", feature_grad_mult=fgm, trainable=True, attention_dropout=0.0,
                                               **SETTINGS["off"]))
        m.remove_pretraining_modules()
        m = m.to(dev, torch.bfloat16).train()
        params = m.full_parameters(True, True)[0] if fgm > 0 else m.tail_parameters()

        def step():
            y, _ = m.extract_finetune({"audio": a, "video": v}, None)
            y.float().pow(2).mean().backward()
            for p in params:
                p.grad = None
            return m._last_train_args[1]

        times = {k: [] for k in SETTINGS}
        dropped = {k: 0 for k in SETTINGS}
        launches = {}
        with torch.cuda.stream(stream):
            for name, reg in SETTINGS.items():      # warm-up: first run, graph capture, replay of every plan
                for key, val in reg.items():
                    setattr(m.cfg, key, val)
                for _ in range(3):
                    step()
                torch.cuda.synchronize(dev)
                _lib.reset_launch_count()
                step()
                torch.cuda.synchronize(dev)
                launches[name] = _lib.launch_count()
            for _ in range(args.rounds):
                for name, reg in SETTINGS.items():
                    for key, val in reg.items():
                        setattr(m.cfg, key, val)
                    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    t0.record()
                    for _ in range(args.steps):
                        dropped[name] += sum(step())
                    t1.record()
                    torch.cuda.synchronize(dev)
                    times[name].append(t0.elapsed_time(t1) / args.steps)
        med = {k: float(np.median(t)) for k, t in times.items()}
        result[f"fgm_{fgm}"] = {
            "ms_per_step_median": med, "ms_per_step_all": times, "launches_per_step": launches,
            "overhead_vs_off_pct": {k: 100.0 * (med[k] / med["off"] - 1.0) for k in med},
            "layers_dropped_per_step": {k: dropped[k] / (args.rounds * args.steps) for k in dropped},
        }
        del m, params
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if "all" not in kk})
                      for k, v in result.items()}, indent=1))


if __name__ == "__main__":
    main()
