#!/usr/bin/env python
"""What switching between training and evaluation costs on one model (Large, 8 clips x 150 frames, bf16 module,
loss = mean(y^2), an SGD update after every training step): the first eval forward after a training step, and the first
training step after that eval, each timed with a host clock around work that ends in a device synchronise.

  device  the switch as the library does it: the first eval forward refreshes the eval-only packed forms (and the
          training forms, for the update since the last training forward) in place on the device; handle, plans and
          captured graphs stay
  repack  the switch through the host, forced with refresh_weights() before the eval forward: every state-dict tensor
          copied to the host, packed, uploaded, and every plan, arena and graph dropped (so the training step after
          the eval rebuilds and re-captures its plans)

Both modes alternate in one process on a non-default stream; the steady eval forward and training step of the same
model are timed for reference.
  python tools/train_eval_switch.py [--fgm 0.0] [--rounds R] [--out profiles/train_eval_switch.json]      (needs a B200)"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fgm", type=float, default=0.0, help="feature_grad_mult: 0 = frozen extractors, 1 = whole model")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "train_eval_switch.json"))
    args = ap.parse_args()
    import numpy as np
    import torch
    from multimodalvc_b200 import AVHubertConfig, AVHubertModel
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(500)
    src = {"video": torch.randn(8, 1, 150, 88, 88, generator=g).to(dev, torch.bfloat16),
           "audio": torch.randn(8, 104, 150, generator=g).to(dev, torch.bfloat16)}
    np.random.seed(0)
    torch.manual_seed(0)
    m = AVHubertModel(AVHubertConfig.named("large", feature_grad_mult=args.fgm, trainable=True, attention_dropout=0.0,
                                           dropout_input=0.0, dropout=0.0, activation_dropout=0.0, encoder_layerdrop=0.0))
    m.remove_pretraining_modules()
    m = m.to(dev, torch.bfloat16).train()
    opt = torch.optim.SGD([p for p in m.parameters() if p.requires_grad], lr=1e-6)
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))

    def clock(fn):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(dev)
        return 1e3 * (time.perf_counter() - t0)

    def train_step():
        opt.zero_grad(set_to_none=True)
        y, _ = m.extract_finetune(src, None)
        y.float().pow(2).mean().backward()

    def eval_forward():
        with torch.no_grad():
            m.extract_finetune(src, None)

    times = {"device": {"first_eval_ms": [], "first_train_step_ms": []},
             "repack": {"first_eval_ms": [], "first_train_step_ms": []}}
    steady = {"eval_ms": [], "train_step_ms": []}
    with torch.cuda.stream(stream):
        for _ in range(3):                      # warm-up: plan build, graph capture, replay
            train_step(); opt.step()
        m.eval()
        for _ in range(3):
            eval_forward()
        m.train()
        for _ in range(args.rounds):
            for mode in ("device", "repack"):
                train_step()
                opt.step()
                if mode == "repack":
                    m.refresh_weights()
                m.eval()
                times[mode]["first_eval_ms"].append(clock(eval_forward))
                t = clock(eval_forward)
                if mode == "device":               # after a re-pack the second run captures the eval plan's graphs
                    steady["eval_ms"].append(t)
                m.train()
                times[mode]["first_train_step_ms"].append(clock(train_step))
                opt.step()
                train_step()                    # the plan is captured on its second run
                opt.step()
                t = clock(train_step)
                if mode == "device":
                    steady["train_step_ms"].append(t)
                opt.step()
    med = lambda xs: float(np.median(xs))
    result = {"card": card(), "shape": "large, 8 x 150, bf16 module", "feature_grad_mult": args.fgm, "rounds": args.rounds,
              "median_ms": {mode: {k: med(v) for k, v in d.items()} for mode, d in times.items()},
              "steady_median_ms": {k: med(v) for k, v in steady.items()},
              "all_ms": {"modes": times, "steady": steady}}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "all_ms"}, indent=1))


if __name__ == "__main__":
    main()
