#!/usr/bin/env python
"""What one AV-HuBERT pretraining step costs on the device (Large, 8 clips x 150 frames, bf16 module, final_dim 256, one
dictionary of V classes, span masking, loss = the criterion's cross-entropies + 10 * features_pen), alternating in one
process on a non-default stream:

  pretrain       AVHubertModel.forward in .train() + backward, no modality dropped
  pretrain_video the same step with the video modality dropped (its ResNet forward still runs, its backward is skipped)
  finetune       extract_finetune in .train() + backward of mean(y^2) on the same model (BASELINE config 5's step)
  head           final_proj + the cosine logits, forward + backward alone on [1200, 1024] encoder rows (CUDA events)

Steps are timed with a host clock around work that ends in a device synchronise; the card's name, power limit and
maximum SM clock are printed beside the numbers.
  python tools/pretrain_step.py --classes 500 [--fgm 0.1] [--rounds 5] [--out result.json]      (needs a B200)"""
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
    ap.add_argument("--classes", type=int, default=500, help="V, the dictionary size")
    ap.add_argument("--fgm", type=float, default=0.1, help="feature_grad_mult (0.1 in the shipped pretraining configs)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import types
    import numpy as np
    import torch
    import torch.nn.functional as F
    from multimodalvc_b200 import AVHubertConfig, AVHubertModel
    from multimodalvc_b200.hubert import _LogitsFn
    dev = torch.device("cuda", 0)
    B, T, V = 8, 150, args.classes
    g = torch.Generator().manual_seed(500)
    src = {"video": torch.randn(B, 1, T, 88, 88, generator=g).to(dev, torch.bfloat16),
           "audio": torch.randn(B, 104, T, generator=g).to(dev, torch.bfloat16)}
    pm = torch.zeros(B, T, dtype=torch.bool, device=dev)
    targets = [torch.randint(0, V, (B, T), generator=g).to(dev)]
    np.random.seed(0)
    torch.manual_seed(0)
    cfg = AVHubertConfig.named("large", feature_grad_mult=args.fgm, trainable=True, attention_dropout=0.0, dropout_input=0.0,
                               dropout=0.0, activation_dropout=0.0, encoder_layerdrop=0.0, final_dim=256,
                               modality_dropout=0.0, audio_dropout=0.0)
    m = AVHubertModel(cfg, types.SimpleNamespace(sample_rate=25), [list(range(V))]).to(dev, torch.bfloat16).train()
    stream = torch.cuda.Stream(device=dev)
    stream.wait_stream(torch.cuda.current_stream(dev))

    def clock(fn):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(dev)
        return 1e3 * (time.perf_counter() - t0)

    def pretrain(drop_video):
        m.cfg.modality_dropout = 1.0 if drop_video else 0.0     # the coins still drawn; a probability of 1 always drops
        m.zero_grad(set_to_none=True)
        res = m(src, target_list=targets, padding_mask=pm, mask=True)
        loss = 10.0 * res["features_pen"]
        for lm, lu, tm, tu in zip(res["logit_m_list"], res["logit_u_list"], res["target_m_list"], res["target_u_list"]):
            loss = loss + F.cross_entropy(lm, tm, reduction="sum") + F.cross_entropy(lu, tu, reduction="sum")
        loss.backward()

    def finetune():
        m.zero_grad(set_to_none=True)
        y, _ = m.extract_finetune(src, pm)
        y.float().pow(2).mean().backward()

    x = torch.randn(B * T, 1024, generator=g).to(dev, torch.bfloat16).requires_grad_(True)
    W = m.final_proj.weight
    bias = m.final_proj.bias
    E = m.label_embs_concat

    def head():
        proj = _LogitsFn.apply(x, W, bias, 0, 1.0)
        _LogitsFn.apply(proj, E, None, 1, 0.1).sum().backward()

    steps = {"pretrain": lambda: pretrain(False), "pretrain_video": lambda: pretrain(True), "finetune": finetune}
    times = {k: [] for k in steps}
    head_ms = []
    with torch.cuda.stream(stream):
        for fn in steps.values():             # warm-up: plan build, graph capture, replay
            for _ in range(3):
                fn()
        for _ in range(10):
            head()
        for _ in range(args.rounds):
            for k, fn in steps.items():
                times[k].append(clock(fn))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(20):
                head()
            e1.record(stream)
            e1.synchronize()
            head_ms.append(e0.elapsed_time(e1) / 20)
    med = lambda xs: float(np.median(xs))
    flops_head = 2.0 * 3 * B * T * (1024 * 256 + 256 * V)      # forward + both backward contractions, both linears
    result = {"card": card(), "shape": f"large, {B} x {T}, bf16 module, final_dim 256, V {V}, feature_grad_mult {args.fgm}",
              "rounds": args.rounds, "median_ms": {k: med(v) for k, v in times.items()}, "head_median_ms": med(head_ms),
              "head_share_of_pretrain_step": med(head_ms) / med(times["pretrain"]), "head_gflop": flops_head / 1e9,
              "all_ms": {**times, "head": head_ms}}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "all_ms"}, indent=1))


if __name__ == "__main__":
    main()
