#!/usr/bin/env python
"""bench.py — AV-HuBERT-Large encoder 6 s-clips/sec on N B200s (BASELINE.json metric), one JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path (AVHubertModel.extract_finetune, audio+video) over one batch of
16 synthetic 6 s clips (150 frames of 88x88 + 104-dim stacked log-fbank features) per GPU, bf16 operands /
fp32 accumulation, random-init Large weights (BASELINE config 2).  Ranks shard clips with no data-path
collective (weak scaling); the timed region is bracketed by barrier + synchronize and the max over ranks is
taken.  `value` has inputs resident in HBM; `e2e` goes through avh_forward_host with pinned HOST buffers
(H2D of the inputs and D2H of the features inside the timed region).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B_PER_GPU, T_FRAMES, N_ROTATE = 16, 150, 4
D, F, L, H = 1024, 4096, 24, 16
METRIC = "AV-HuBERT-L encoder 6s-clips/sec"
UNIT = "clips/s"

FRONTEND_MAC = 316_158_976                     # per video frame (BASELINE.md §3)


def clip_flops(T=T_FRAMES, audio=True):
    """Algorithmic FLOPs (2*MAC) of one clip: (total, attention part)."""
    lin = 512 * D + (104 * D if audio else 0) + 2 * D * D + D * (D // 16) * 128 + L * (4 * D * D + 2 * D * F)
    att = L * 2 * T * D
    mac = T * (FRONTEND_MAC + lin + att)
    return 2.0 * mac, 2.0 * T * att


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons (NVML, ~2 ms period; same fields as the nvidia-smi clocks line of
    B200_PROFILING.md).  Runs from before the warm-up; `summary(t0, t1)` reports the samples taken inside a timed
    region (host perf_counter window around the synchronised region)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.max_sm, self.stop_flag, self.ready = index, [], None, False, threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if visible:
                try:
                    idx = int(visible.split(",")[self.index])
                except Exception:
                    pass
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            self.ready.set()
            while not self.stop_flag:
                self.samples.append((time.perf_counter(), pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM),
                                     int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))))
                time.sleep(float(os.environ.get('AVH_BENCH_SAMPLE_S', '0.002')))
        except Exception as e:      # clocks are evidence, not part of the measurement: never fail the run
            self.err = str(e)
            self.ready.set()

    def summary(self, t0=None, t1=None):
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        sel = [x for x in self.samples if (t0 is None or x[0] >= t0) and (t1 is None or x[0] <= t1)]
        note = None
        if not sel and self.samples and t0 is not None:      # region shorter than the sampling period: nearest sample
            sel = [min(self.samples, key=lambda x: abs(x[0] - 0.5 * (t0 + t1)))]
            note = "region shorter than the sampling period: nearest sample"
        sm = sorted(x[1] for x in sel)
        mask = 0
        for x in sel:
            mask |= x[2]
        out = {"sm_mhz": float(sm[len(sm) // 2]) if sm else None, "sm_min_mhz": float(sm[0]) if sm else None,
               "sm_max_mhz": float(self.max_sm) if self.max_sm else None,
               "reasons": sorted(v for k, v in names.items() if mask & k), "samples": len(sm)}
        if note:
            out["note"] = note
        return out


def _parse_cpulist(txt):
    cpus = []
    for part in txt.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.extend(range(int(a), int(b or a) + 1))
    return cpus


def pin_host_thread(local_rank, world):
    """Bind this rank's host thread (and, by first touch, its pinned buffers) to cores of the GPU's own NUMA node:
    with 8 ranks x 3 streams of pinned H2D/D2H, unpinned ranks all sat on NUMA node 0 (r1: e2e efficiency 0.937 at
    N=8 against 0.978 device-resident).  The node's cores are split evenly between the ranks whose GPUs share it."""
    info = {"pinned": False}
    try:
        import torch
        props = [torch.cuda.get_device_properties(i) for i in range(torch.cuda.device_count())]

        def sysfs(pr):
            return f"/sys/bus/pci/devices/{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        nodes = []
        for pr in props:
            try:
                nodes.append(int(open(sysfs(pr) + "/numa_node").read()))
            except Exception:
                nodes.append(-1)
        node = nodes[local_rank]
        cpus = _parse_cpulist(open(sysfs(props[local_rank]) + "/local_cpulist").read())
        allowed = sorted(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed] or allowed
        peers = [i for i in range(min(world, len(nodes))) if nodes[i] == node]
        k = peers.index(local_rank) if local_rank in peers else 0
        share = max(1, len(cpus) // max(1, len(peers)))
        mine = cpus[k * share:(k + 1) * share] or cpus
        os.sched_setaffinity(0, mine)
        info = {"pinned": True, "numa_node": node, "cpus": f"{mine[0]}-{mine[-1]}", "n_cpus": len(mine)}
    except Exception as e:      # placement is an optimisation: never fail the run
        info["error"] = str(e)[:120]
    return info


def synthetic_wave(n_samples, seed):
    """Synthetic 16 kHz int16 audio of SURVEY 8(d): clip(round(3000 * randn)).  (Defined here so that the product arm
    of the bench imports nothing from oracle/.)"""
    import numpy as np
    r = np.random.RandomState(seed)
    return np.clip(np.round(3000.0 * r.randn(n_samples)), -32768, 32767).astype(np.int16)


def hbm_kernels(dev, prof):
    """Achieved algorithmic GB/s of the HBM-bound kernels north_star names (log-fbank, noise mixing, LayerNorm),
    CUDA events on the launching stream, inputs larger than L2 (256 clips x 6 s = 49 MB of int16 samples)."""
    import torch
    from multimodalvc_b200 import audio
    n_clips, n_samp = 256, T_FRAMES * 640
    g = torch.Generator().manual_seed(5)
    flat = (torch.randn(n_clips * n_samp, generator=g) * 3000).clamp(-32768, 32767).to(torch.int16).to(dev)
    off = (torch.arange(n_clips + 1, dtype=torch.int64) * n_samp).to(dev)
    vlen = torch.full((n_clips,), T_FRAMES, dtype=torch.int32, device=dev)
    wavs = [flat[i * n_samp:(i + 1) * n_samp] for i in range(n_clips)]
    noise = torch.randn(100000, generator=g).mul(2000).to(dev)

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize(dev)
        best = 1e30
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            best = min(best, a.elapsed_time(b))
        return best

    out = []
    ms_f = timed(lambda: audio.logfbank_stack_collate_packed(flat, off, T_FRAMES, vlen))
    by_f = n_clips * (2 * n_samp + 4 * 104 * T_FRAMES)            # SURVEY 8(d): 254 400 B per 6 s clip
    out.append({"kernel": "fbank_kernel (log-fbank + stack + align + LN + collate)", "algorithmic_bytes": by_f,
                "ms": ms_f, "achieved": by_f / (ms_f * 1e-3) / 1e9, "unit": "GB/s",
                "note": "one 512-point real FFT in float64 per 10 ms frame: FP64-ALU / shared-memory bound, not HBM bound"})
    ms_n = timed(lambda: audio.add_noise_packed(flat, off, noise, 0.0))
    by_n = n_clips * n_samp * 4                                    # read int16 clean + write int16 mixed
    out.append({"kernel": "noise_* (add_noise: RMS sums, min/max, mix + int16 truncation; 3 passes + init)",
                "algorithmic_bytes": by_n, "ms": ms_n, "achieved": by_n / (ms_n * 1e-3) / 1e9, "unit": "GB/s",
                "note": "the clean waveform is read three times (two reductions feed the scale and the clip rescale)"})
    ln = prof.get("layer_ln")
    if ln and ln["launches"]:
        by_l = B_PER_GPU * T_FRAMES * D * (4 + 2)                  # fp32 residual stream in, bf16 operand out
        ms_l = ln["ms"] / ln["launches"]
        out.append({"kernel": "layernorm_f32_vec_kernel (per-layer LayerNorm)", "algorithmic_bytes": by_l, "ms": ms_l,
                    "achieved": by_l / (ms_l * 1e-3) / 1e9, "unit": "GB/s", "launches_per_step": ln["launches"],
                    "note": "14.7 MB per launch: latency-bound (one wave of 600 CTAs), input L2-resident in the pipeline"})
    return out


def build_oracle_large(threads):
    import torch
    from oracle import avhubert_oracle as ao
    torch.set_num_threads(threads)
    return ao.build_oracle("large", seed=1234)


def time_oracle(oracle, B, steps, warmup):
    """CPU forward of the fp32 oracle (restatement of the reference's PyTorch path) on B clips."""
    import torch
    from oracle import avhubert_oracle as ao
    src, _ = ao.synthetic_inputs(B, T_FRAMES, seed=21)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            oracle.extract_finetune(src, None)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    return times


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path.  The reference is Python and
    /root/reference does not travel to the GPU box, so this is the oracle port (pinned against the real
    reference in tests/), with all host threads, on the bench workload: the whole 16-clip batch per step when
    K + W such steps fit in ~4 minutes, else the largest number of clips per step that does (stated in `sample`)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    oracle = build_oracle_large(cores)
    warm = max(1, min(args.warmup, 2))
    steps = max(1, args.steps)
    t_probe = time_oracle(oracle, 2, 1, 1)[0]                 # s for 2 clips (after one warm-up forward)
    budget = 240.0
    sample_b = B_PER_GPU
    while sample_b > 1 and (t_probe / 2.0) * sample_b * (steps + warm) > budget:
        sample_b //= 2
    times = time_oracle(oracle, sample_b, steps, warm)
    total = sum(times)
    value = sample_b * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": warm, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE config 2: AV-HuBERT Large (24L, d=1024) extract_finetune, audio+video, "
                               "batch 16 x 6 s clips (150 frames) per GPU, random-init weights",
                   "per_gpu_batch": B_PER_GPU, "frames": T_FRAMES, "clips_per_timed_forward": sample_b},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{sample_b} of the {B_PER_GPU} clips of a step per timed forward "
                                   f"({'the whole batch' if sample_b == B_PER_GPU else 'bounded so the run ends within minutes'}), "
                                   "fp32 PyTorch CPU oracle (restatement of the reference path; the Python reference "
                                   "cannot travel to the GPU box)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streams", type=int, default=3,
                    help="CUDA streams per GPU; consecutive steps alternate between them (each has its own workspace)")
    ap.add_argument("--sustain-s", type=float, default=3.0,
                    help="seconds of back-to-back steps for the `sustained` leg after the timed region (0 = skip)")
    ap.add_argument("--config3-passes", type=int, default=5, help="timed passes over the 64 ragged clips of config 3 (0 = skip)")
    ap.add_argument("--config3-tokens", type=int, default=4800, help="packed frames per ragged sub-batch")
    ap.add_argument("--config4-passes", type=int, default=2,
                    help="timed passes over the 32 noisy 24 s clips of BASELINE config 4 (0 = skip)")
    ap.add_argument("--config5-steps", type=int, default=5,
                    help="timed fine-tuning steps of BASELINE config 5 (forward + backward + gradient all-reduce; 0 = skip)")
    ap.add_argument("--profile-json", default=None, help="write the per-kernel-class breakdown here")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the features the last timed step returned (rank 0) as DIR/features.npy, float32, so that "
                         "two builds can be compared output for output (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from multimodalvc_b200 import AVHubertConfig, AVHubertModel, _lib, audio
    from multimodalvc_b200 import build as avh_build

    if not torch.cuda.is_available():
        sys.exit("bench.py needs a B200: the product path has no CPU fallback")
    avh_build.build()
    args.warmup = max(args.warmup, 3)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    full_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    # AVH_BENCH_PIN=0 leaves placement to the OS; the CPU-baseline leg gets every core back (below)
    affinity = (pin_host_thread(local_rank, world) if os.environ.get("AVH_BENCH_PIN", "1") != "0"
                else {"pinned": False, "note": "AVH_BENCH_PIN=0: left to the OS"})
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL announces its version on stdout at the first collective; stdout carries exactly ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- model: random-init Large weights (same seed on every rank), bf16 compute
    torch.manual_seed(1234)
    model = AVHubertModel(AVHubertConfig.named("large", frontend_chunk_frames=int(os.environ.get("AVH_BENCH_CHUNK", "0"))))
    model.remove_pretraining_modules()
    model = model.to(dev, torch.bfloat16).eval()

    # ---- synthetic inputs: N_ROTATE distinct batches so no step finds its inputs in L2 from the previous one
    g = torch.Generator().manual_seed(100 + rank)
    host_v, host_a, dev_v, dev_a = [], [], [], []
    for r in range(N_ROTATE):
        v = torch.randn(B_PER_GPU, 1, T_FRAMES, 88, 88, generator=g).to(torch.bfloat16)
        wavs = [torch.from_numpy(synthetic_wave(T_FRAMES * 640, 1000 * rank + 16 * r + i)) for i in range(B_PER_GPU)]
        a, _ = audio.logfbank_stack_collate(wavs, video_lens=[T_FRAMES] * B_PER_GPU, device=dev)
        a = a.to(torch.bfloat16)
        host_v.append(v.pin_memory())
        host_a.append(a.contiguous().cpu().pin_memory())
        dev_v.append(v.to(dev))
        dev_a.append(a)
    S = max(1, args.streams)
    host_out = [torch.empty(B_PER_GPU, T_FRAMES, D, dtype=torch.bfloat16).pin_memory() for _ in range(S)]
    streams = [torch.cuda.Stream(dev) for _ in range(S)]
    main_stream = torch.cuda.current_stream(dev)

    def step(i):
        with torch.cuda.stream(streams[i % S]):
            return model.extract_finetune({"audio": dev_a[i % N_ROTATE], "video": dev_v[i % N_ROTATE]}, None)[0]

    def step_host(i):
        st = streams[i % S]
        st.synchronize()            # the previous result in this stream's host buffer has been read back
        with torch.cuda.stream(st):
            return model.extract_finetune_host(host_v[i % N_ROTATE], host_a[i % N_ROTATE], None, out=host_out[i % S],
                                               wait=False)

    def fork(evt):
        for st in streams:
            st.wait_event(evt)

    def join():
        for st in streams:
            main_stream.wait_stream(st)

    # ---- device-resident timing
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.ready.wait(timeout=10)
    torch.cuda.synchronize(dev)
    # warm-up: at least W steps, and enough for every (stream, input batch) pair to have been seen twice — the library
    # runs the first call of a shape directly and captures a CUDA graph per distinct set of input pointers on the
    # next ones; with fewer warm-up steps those one-off captures (ms of host time each) fall into the timed region
    n_warm = max(args.warmup, S * N_ROTATE + S)
    for i in range(n_warm):
        step(i)
    join()
    barrier()
    _lib.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_region0 = time.perf_counter()
    e0.record()
    fork(e0)
    for i in range(args.steps):
        y = step(i)
    join()
    e1.record()
    barrier()
    t_region1 = time.perf_counter()
    launches = _lib.launch_count()
    ms = e0.elapsed_time(e1)
    clocks_timed = sampler.summary(t_region0, t_region1)
    checksum = float(y.float().abs().mean().item())
    if args.dump_outputs and rank == 0:
        # [16, 150, 1024] bf16 -> float32 (exact), 9.8 MB; the padding mask extract_finetune returns is None here
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "features.npy"), y.float().cpu().numpy())

    # ---- sustained leg: >= SUSTAIN_S seconds of back-to-back steps (the driver-sized region above is ~0.1 s, i.e.
    #      burst clocks); reports what the power cap does to the rate over seconds
    sustained = None
    if args.sustain_s > 0:
        n_sus = max(args.steps, int(args.sustain_s / max(ms / args.steps * 1e-3, 1e-4)) + 1)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_sus0 = time.perf_counter()
        s0.record()
        fork(s0)
        for i in range(n_sus):
            step(i)
        join()
        s1.record()
        barrier()
        ms_sus = s0.elapsed_time(s1)
        sustained = (n_sus, ms_sus, sampler.summary(t_sus0, time.perf_counter()))
    sampler.stop_flag = True
    sampler.join(timeout=3)

    # ---- end to end through the host-buffer entry point
    for i in range(2 * S):
        step_host(i)
    join()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    fork(f0)
    for i in range(args.steps):
        step_host(i)
    join()
    f1.record()
    barrier()              # every D2H copy has landed in pinned host memory
    ms_e2e = f0.elapsed_time(f1)

    # ---- the same end-to-end call fed with RAW uint8 mouth-ROI frames (96 x 96, as the dataset stores them): the
    #      /255 -> centre crop -> (x-mean)/std transform runs on the device (SURVEY 8(f)-1), 1 byte per pixel over PCIe
    host_u8 = [torch.randint(0, 256, (B_PER_GPU, 1, T_FRAMES, 96, 96), dtype=torch.uint8, generator=g).pin_memory()
               for _ in range(N_ROTATE)]

    def step_host_u8(i):
        st = streams[i % S]
        st.synchronize()
        with torch.cuda.stream(st):
            return model.extract_finetune_host(host_u8[i % N_ROTATE], host_a[i % N_ROTATE], None, out=host_out[i % S],
                                               wait=False)

    for i in range(2 * S):
        step_host_u8(i)
    join()
    barrier()
    u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u0.record()
    fork(u0)
    for i in range(args.steps):
        step_host_u8(i)
    join()
    u1.record()
    barrier()
    ms_e2e_u8 = u0.elapsed_time(u1)

    # ---- the WHOLE path of SURVEY 8(a) from raw host inputs: uint8 frames + int16 waveforms (pinned) -> H2D ->
    #      log-fbank/stack/LN/collate kernel (A1-A6) -> frame transform + encoder (A7-A17) -> D2H of the features
    n_samp = T_FRAMES * 640
    host_wav = [torch.cat([torch.from_numpy(synthetic_wave(n_samp, 5000 * rank + 16 * r + i)) for i in range(B_PER_GPU)])
                .pin_memory() for r in range(N_ROTATE)]
    wav_off = (torch.arange(B_PER_GPU + 1, dtype=torch.int64) * n_samp).to(dev)
    vlen = torch.full((B_PER_GPU,), T_FRAMES, dtype=torch.int32, device=dev)
    dev_wav = [torch.empty_like(host_wav[0], device=dev) for _ in range(S)]
    dev_u8 = [torch.empty_like(host_u8[0], device=dev) for _ in range(S)]

    def step_raw_av(i):
        st = streams[i % S]
        st.synchronize()
        with torch.cuda.stream(st):
            dev_wav[i % S].copy_(host_wav[i % N_ROTATE], non_blocking=True)
            dev_u8[i % S].copy_(host_u8[i % N_ROTATE], non_blocking=True)
            a, _ = audio.logfbank_stack_collate_packed(dev_wav[i % S], wav_off, T_FRAMES, vlen)
            yy = model.extract_finetune({"audio": a, "video": dev_u8[i % S]}, None)[0]
            host_out[i % S].copy_(yy, non_blocking=True)

    for i in range(2 * S):
        step_raw_av(i)
    join()
    barrier()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    fork(r0)
    for i in range(args.steps):
        step_raw_av(i)
    join()
    r1.record()
    barrier()
    ms_e2e_raw = r0.elapsed_time(r1)

    # ---- BASELINE config 3: 64 ragged clips (U{25..600} frames, seed 7) with key-padding masks, sharded over the ranks
    #      (balanced_shards), each rank running its clips as packed sub-batches (cfg.ragged='packed': no work on pad
    #      frames).  Device-resident inputs; one "pass" = all 64 clips once.
    cfg3 = None
    if args.config3_passes > 0:
        from multimodalvc_b200 import sharding
        g3 = torch.Generator().manual_seed(7)
        lengths3 = torch.randint(25, 601, (64,), generator=g3).tolist()
        mine = sharding.balanced_shards(lengths3, world)[rank]
        subs = sharding.token_buckets(mine, lengths3, max_tokens=args.config3_tokens, max_clips=32)
        gin = torch.Generator().manual_seed(300 + rank)
        batches = []
        for sb in subs:
            tb = max(lengths3[i] for i in sb)
            v3 = torch.zeros(len(sb), 1, tb, 88, 88, dtype=torch.bfloat16)
            a3 = torch.zeros(len(sb), 104, tb, dtype=torch.bfloat16)
            pm3 = torch.ones(len(sb), tb, dtype=torch.bool)
            for j, i in enumerate(sb):
                n = lengths3[i]
                v3[j, :, :n] = torch.randn(1, n, 88, 88, generator=gin).to(torch.bfloat16)
                a3[j, :, :n] = torch.randn(104, n, generator=gin).to(torch.bfloat16)
                pm3[j, :n] = False
            batches.append((v3.to(dev), a3.to(dev), pm3.to(dev), [lengths3[i] for i in sb]))
        model.cfg.ragged = "packed"

        def pass3(k):
            for j, (v3, a3, pm3, ln3) in enumerate(batches):
                with torch.cuda.stream(streams[(k * len(batches) + j) % S]):
                    model.extract_finetune({"audio": a3, "video": v3}, pm3, lengths=ln3)

        for k in range(3):
            pass3(k)
        join()
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        fork(c0)
        for k in range(args.config3_passes):
            pass3(k)
        join()
        c1.record()
        barrier()
        model.cfg.ragged = "dense"
        frames_mine = sum(lengths3[i] for i in mine)
        padded_dense = sum(len(sb) * max(lengths3[i] for i in sb) for sb in subs)
        cfg3 = {"ms": c0.elapsed_time(c1), "frames_all": sum(lengths3), "frames_rank0": frames_mine,
                "sub_batches_rank0": [[len(sb), sum(lengths3[i] for i in sb)] for sb in subs],
                "pad_fraction_if_dense_rank0": 1.0 - frames_mine / float(padded_dense)}

    # ---- BASELINE config 4: noisy evaluation — 32 clips x 24 s (600 frames) per GPU, babble noise mixed at -5 / 0 / 5 dB
    #      on the device (add_noise), log-fbank + stack + LayerNorm + collate (avh_fbank), then the Large forward, as 4
    #      sub-batches of 8 clips (4800 frames each).  Waveforms, noise and uint8 frames device-resident.
    cfg4 = None
    if args.config4_passes > 0:
        from multimodalvc_b200 import audio as avh_audio
        import numpy as np
        T4, NB4, SUB4 = 600, 32, 8
        r4 = np.random.RandomState(400 + rank)
        babble = np.mean([np.clip(np.round(3000.0 * r4.randn(T4 * 640)), -32768, 32767) for _ in range(30)], axis=0)
        noise4 = torch.from_numpy(babble.astype(np.float32)).to(dev)
        subs4 = []
        for j in range(NB4 // SUB4):
            wav = torch.from_numpy(np.clip(np.round(3000.0 * r4.randn(SUB4 * T4 * 640)), -32768, 32767).astype(np.int16)).to(dev)
            offs = (torch.arange(SUB4 + 1, dtype=torch.int64) * (T4 * 640)).to(dev)
            vid = torch.randint(0, 256, (SUB4, 1, T4, 88, 88), dtype=torch.uint8,
                                generator=torch.Generator().manual_seed(410 + rank * 8 + j)).to(dev)
            subs4.append((wav, offs, vid, (-5.0, 0.0, 5.0, 0.0)[j]))

        def pass4(k):
            for j, (wav, offs, vid, snr) in enumerate(subs4):
                with torch.cuda.stream(streams[(k * len(subs4) + j) % S]):
                    mixed = avh_audio.add_noise_packed(wav, offs, noise4, snr)
                    a4, _ = avh_audio.logfbank_stack_collate_packed(mixed, offs, T4)
                    model.extract_finetune({"audio": a4.to(torch.bfloat16), "video": vid}, None)

        for k in range(2):
            pass4(k)
        join()
        barrier()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        fork(d0)
        for k in range(args.config4_passes):
            pass4(k)
        join()
        d1.record()
        barrier()
        cfg4 = {"ms": d0.elapsed_time(d1)}
        del subs4

    # ---- BASELINE config 5: Large, B = 8 clips x 150 frames per GPU, bf16, dropout / LayerDrop 0, loss = mean(x^2);
    #      forward + backward + gradient all-reduce per step.  Two forms: the whole model differentiable
    #      (feature_grad_mult = 0.1: lip ResNet, projections, encoder) and the frozen-extractor form (feature_grad_mult = 0,
    #      the reference then runs the extractors under no_grad).
    cfg5 = None
    cfg5_frozen = None
    cfg5_opt = None
    if args.config5_steps > 0:
        from multimodalvc_b200.distributed import GradientAllReducer
        g5 = torch.Generator().manual_seed(500 + rank)
        v5 = torch.randn(8, 1, T_FRAMES, 88, 88, generator=g5).to(dev, torch.bfloat16)
        a5 = torch.randn(8, 104, T_FRAMES, generator=g5).to(dev, torch.bfloat16)

        def config5_leg(fgm, with_optimizer=False):
            m5 = AVHubertModel(AVHubertConfig.named("large", feature_grad_mult=fgm, trainable=True, dropout=0.0,
                                                    attention_dropout=0.0, activation_dropout=0.0, encoder_layerdrop=0.0,
                                                    dropout_input=0.0))
            m5.remove_pretraining_modules()
            m5 = m5.to(dev, torch.bfloat16).train()
            params = m5.full_parameters(True, True)[0] if fgm > 0 else m5.tail_parameters()
            reducer = GradientAllReducer(params).attach(m5) if world > 1 else None      # buckets reduced during the backward
            opt5 = torch.optim.SGD(params, lr=1e-5, momentum=0.9) if with_optimizer else None

            def step5():
                y5, _ = m5.extract_finetune({"audio": a5, "video": v5}, None)
                loss = y5.float().pow(2).mean()
                loss.backward()
                if reducer is not None:
                    reducer.all_reduce_grads()
                if opt5 is not None:
                    opt5.step()          # the next forward refreshes the packed weights on the device (avh_refresh_weights_device)
                return loss

            for _ in range(3):
                step5()
                for p5 in params:
                    p5.grad = None
            torch.cuda.synchronize(dev)
            barrier()
            _lib.reset_launch_count()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.config5_steps):
                loss5 = step5()
                for p5 in params:
                    p5.grad = None
            t1.record()
            torch.cuda.synchronize(dev)
            barrier()
            out = {"ms": t0.elapsed_time(t1), "loss": float(loss5.item()),
                   "grad_elements": int(sum(p5.numel() for p5 in params)),
                   "launches_per_step": int(_lib.launch_count()) // args.config5_steps,
                   "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9}
            del m5, reducer, params, opt5
            torch.cuda.empty_cache()
            return out

        s5 = torch.cuda.Stream(device=dev)       # a real stream: the library replays its launch lists as CUDA graphs there
        s5.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s5):
            cfg5 = config5_leg(0.1)
            cfg5_opt = config5_leg(0.1, with_optimizer=True)
            cfg5_frozen = config5_leg(0.0)
        torch.cuda.current_stream(dev).wait_stream(s5)

    # ---- max over ranks
    ms_sus = sustained[1] if sustained else 0.0
    if world > 1:
        t = torch.tensor([ms, ms_e2e, ms_e2e_u8, ms_e2e_raw, ms_sus, cfg3["ms"] if cfg3 else 0.0,
                          cfg5["ms"] if cfg5 else 0.0, cfg4["ms"] if cfg4 else 0.0,
                          cfg5_frozen["ms"] if cfg5_frozen else 0.0, cfg5_opt["ms"] if cfg5_opt else 0.0],
                         device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e, ms_e2e_u8, ms_e2e_raw, ms_sus, ms_c3, ms_c5, ms_c4, ms_c5f, ms_c5o = t.tolist()
        if cfg5_frozen:
            cfg5_frozen["ms"] = ms_c5f
        if cfg5_opt:
            cfg5_opt["ms"] = ms_c5o
        if cfg4:
            cfg4["ms"] = ms_c4
        if cfg3:
            cfg3["ms"] = ms_c3
        if cfg5:
            cfg5["ms"] = ms_c5
        lt = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(lt)
        launches = int(lt.item())

    # ---- per-kernel-class breakdown (CUDA events around every launch, separate instrumented forward)
    prof = model.profile_forward({"audio": dev_a[0], "video": dev_v[0]}, None)
    prof = model.profile_forward({"audio": dev_a[1], "video": dev_v[1]}, None)
    hbm = hbm_kernels(dev, prof) if rank == 0 else None
    if world > 1:
        dist.barrier()

    if rank == 0:
        clips = world * B_PER_GPU * args.steps
        value = clips / (ms * 1e-3)
        flops_clip, flops_att = clip_flops()
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        # kernels are timed ALONE (CUDA events around each launch of an instrumented forward break the PDL overlap):
        # the burst figure is the right denominator; whole-step rates are set against burst and sustained
        peak_burst = float(peaks.get("bf16_tflops", 1640.0))
        peak_sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_hbm = float(peaks.get("hbm_gbs", 6500.0))
        peak_src = ("MEASURED_PEAKS.json bf16_tflops (burst: kernels timed alone)" if peaks
                    else "fallback of B200_PROFILING.md (no MEASURED_PEAKS.json): 1.64 PFLOP/s burst, 1.4 sustained, 6.5 TB/s")
        # dominant kernel = gemm_kernel (tcgen05/TMEM/TMA): encoder Linear layers, positional conv, projections.
        # achieved = algorithmic FLOPs of those launches / their summed duration.  The other tensor-core kernels are
        # listed beside it.
        gemm_classes = {"fc1", "fc2", "qkv_proj", "out_proj", "pos_conv", "proj_video", "proj_audio", "post_extract_proj",
                        "ffn"}

        def group(pred):
            sel = [v for k, v in prof.items() if v["tc_flops"] > 0 and pred(k)]
            g_ms = sum(v["ms"] for v in sel)
            g_fl = sum(v["tc_flops"] for v in sel)
            return g_ms, g_fl, sum(v["launches"] for v in sel)

        gemm_ms, gemm_alg, gemm_launches = group(lambda k: k in gemm_classes)
        total_prof_ms = sum(v["ms"] for v in prof.values())
        achieved = gemm_alg / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        others = []
        for name, pred in [("stem_fused_kernel (Conv3d+BN+PReLU+MaxPool, TS-MMA)", lambda k: k == "stem_fused"),
                           ("conv_window_kernel (layer1 3x3 convs)", lambda k: k == "conv3x3_c64"),
                           ("conv_frame_kernel (layers 2-4 convs)",
                            lambda k: (k.startswith("conv") or k == "downsample") and k != "conv3x3_c64"),
                           ("attention kernel (QK^T, softmax, PV)", lambda k: k == "attention")]:
            o_ms, o_fl, o_n = group(pred)
            if o_ms > 0:
                others.append({"kernel": name, "achieved": o_fl / (o_ms * 1e-3) / 1e12, "unit": "TFLOP/s",
                               "frac": o_fl / (o_ms * 1e-3) / 1e12 / peak_burst, "kernel_ms_per_step": o_ms,
                               "launches_per_step": o_n})
        tc_ms = gemm_ms + sum(o["kernel_ms_per_step"] for o in others)
        whole = B_PER_GPU * flops_clip * args.steps / (ms * 1e-3) / 1e12          # per GPU
        traffic, traffic_src = None, None
        try:       # dram__bytes_read.sum + dram__bytes_write.sum per GEMM launch from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_gemm_dram_traffic.json")))
            traffic, traffic_src = float(tj["mean_bytes_per_launch"]), tj.get("source")
        except Exception:
            pass
        for hk in hbm or []:
            hk["peak"] = peak_hbm
            hk["frac"] = hk["achieved"] / peak_hbm

        def leg(ms_leg, h2d, d2h, what):
            return {"value": clips / (ms_leg * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_leg / args.steps, "input": what}

        d2h = host_out[0].numel() * 2
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "BASELINE config 2: AV-HuBERT Large (24L, d=1024) extract_finetune, audio+video, "
                                   "batch 16 x 6 s clips (150 frames) per GPU, random-init weights",
                       "per_gpu_batch": B_PER_GPU, "frames": T_FRAMES, "parallelism": f"batch-sharded x{world}, no collective", "streams_per_gpu": S,
                       "untimed_warmup_steps": n_warm, "host_affinity_rank0": affinity,
                       "l2": f"{N_ROTATE} rotating input batches + 0.65 GB weights + ~1 GB activations per step >> 126 MB L2"},
            # declared end-to-end number: the WHOLE path from raw host inputs (uint8 frames + int16 waveforms), as a
            # data loader would hand them over; the reference moves fp32 tensors (src/eval.py:196-200), 4x the bytes
            "e2e": leg(ms_e2e_raw, host_u8[0].numel() + host_wav[0].numel() * 2, d2h,
                       "uint8 gray frames [16,1,150,96,96] + int16 16 kHz waveforms [16 x 96000] from pinned host memory; "
                       "log-fbank/stack/LayerNorm/collate (avh_fbank), frame normalise + crop and the encoder on the "
                       "device: rows A1-A17 of SURVEY 8(a) in one timed region; features read back to pinned host memory"),
            "e2e_raw_video": leg(ms_e2e_u8, host_u8[0].numel() + host_a[0].numel() * 2, d2h,
                                 "uint8 gray frames [16,1,150,96,96] + precomputed bf16 audio features from pinned host "
                                 "memory (avh_forward_host with AVH_U8 video)"),
            "e2e_features_bf16": leg(ms_e2e, host_v[0].numel() * 2 + host_a[0].numel() * 2, d2h,
                                     "normalised bf16 frames [16,1,150,88,88] + bf16 audio features from pinned host memory "
                                     "(cast outside the timed region; kept for continuity with round 1's `e2e`)"),
            "gpu_launches": launches,
            "clocks": clocks_timed,
            "roofline": {"bound": "tensor",
                         "kernel": "gemm_kernel (tcgen05/TMEM/TMA): encoder Linear layers + positional conv + projections",
                         "achieved": achieved, "peak": peak_burst, "unit": "TFLOP/s", "frac": achieved / peak_burst,
                         "frac_of_sustained_peak": achieved / peak_sus,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "launches_per_step": gemm_launches, "kernel_ms_per_step": gemm_ms,
                         "share_of_step": gemm_ms / total_prof_ms if total_prof_ms else None,
                         "timing": "CUDA events around each launch of an instrumented forward on the launching stream "
                                   "(isolated launches: no PDL overlap, ~+25 % vs the in-pipeline CUPTI timeline of "
                                   "tools/timeline.py)",
                         "other_tensor_kernels": others,
                         "tensor_kernels_share_of_step": tc_ms / total_prof_ms if total_prof_ms else None,
                         "whole_step_tflops_per_gpu": whole,
                         "whole_step_frac_of_burst": whole / peak_burst, "whole_step_frac_of_sustained": whole / peak_sus,
                         "whole_step_frac": whole / peak_sus},
            "roofline_hbm": hbm,
            "output_checksum": checksum,
        }
        if sustained:
            n_sus, _, sus_clk = sustained
            v_sus = world * B_PER_GPU * n_sus / (ms_sus * 1e-3)
            w_sus = B_PER_GPU * flops_clip * n_sus / (ms_sus * 1e-3) / 1e12
            line["sustained"] = {"value": v_sus, "unit": UNIT, "steps": n_sus, "seconds": ms_sus * 1e-3,
                                 "ms_per_step": ms_sus / n_sus, "clocks": sus_clk, "tflops_per_gpu": w_sus,
                                 "frac_of_sustained_peak": w_sus / peak_sus, "frac_of_burst_peak": w_sus / peak_burst}
        if cfg3:
            sec = cfg3["ms"] * 1e-3 / args.config3_passes
            fps3 = cfg3["frames_all"] / sec
            fps2 = value * T_FRAMES
            line["config3"] = {
                "workload": "BASELINE config 3: Large, 64 ragged clips of 25..600 frames (U, seed 7) + key-padding masks, "
                            f"clips dealt to {world} rank(s) by balanced_shards, packed sub-batches of <= "
                            f"{args.config3_tokens} frames (cfg.ragged='packed'), device-resident inputs",
                "clips_per_s": 64.0 / sec, "frames_per_s": fps3, "ms_per_pass": sec * 1e3, "passes": args.config3_passes,
                "frames": cfg3["frames_all"], "config2_frames_per_s": fps2, "frac_of_config2_frame_rate": fps3 / fps2,
                "sub_batches_rank0_clips_frames": cfg3["sub_batches_rank0"],
                "pad_fraction_if_dense_rank0": cfg3["pad_fraction_if_dense_rank0"]}
        if cfg4:
            sec4 = cfg4["ms"] * 1e-3 / args.config4_passes
            fps4 = world * 32 * 600 / sec4
            line["config4"] = {
                "workload": "BASELINE config 4: Large, 32 clips x 24 s (600 frames) per GPU, babble noise mixed at -5 / 0 / 5 dB "
                            "(add_noise on the device), log-fbank + stack + LayerNorm + collate (avh_fbank), uint8 frames "
                            "normalised on the device, forward as 4 sub-batches of 8 clips; device-resident waveforms / frames",
                "clips_per_s": world * 32 / sec4, "frames_per_s": fps4, "ms_per_pass": sec4 * 1e3,
                "passes": args.config4_passes, "config2_frames_per_s": value * T_FRAMES,
                "frac_of_config2_frame_rate": fps4 / (value * T_FRAMES),
                "note": "attention grows with T (600 keys per query instead of 150): 790.5 GFLOP per 24 s clip against "
                        "4 x 190.99 for four 6 s clips"}
        if cfg5:
            sec5 = cfg5["ms"] * 1e-3 / args.config5_steps
            line["config5"] = {
                "workload": "BASELINE config 5: AV-HuBERT Large fine-tuning step with the whole model differentiable "
                            "(feature_grad_mult = 0.1), 8 clips x 150 frames per GPU, bf16, dropout / LayerDrop 0, loss = "
                            "mean(x^2); forward (lip ResNet as patch GEMMs with batch-statistics BatchNorm, projections, "
                            "fusion LayerNorm, post_extract_proj, 24 encoder layers, activations saved) + backward of all of "
                            "it + bucketed gradient all-reduce (NCCL) at N > 1",
                "clips_per_s": world * 8 / sec5, "ms_per_step": sec5 * 1e3, "steps": args.config5_steps,
                "grad_elements": cfg5["grad_elements"], "loss": cfg5["loss"],
                "launches_per_step": cfg5["launches_per_step"], "peak_mem_gb": cfg5["peak_mem_gb"],
                "not_included": "optimizer step (BASELINE config 5 is forward + backward + all-reduce; see "
                                "config5_with_optimizer for the whole iteration)"}
        if cfg5_opt:
            sec5 = cfg5_opt["ms"] * 1e-3 / args.config5_steps
            line["config5_with_optimizer"] = {
                "workload": "config 5 as a whole training iteration: the step above + SGD(momentum) on the bf16 parameters + the "
                            "in-place device-side refresh of the packed weights before the next forward "
                            "(avh_refresh_weights_device; the host re-pack this replaces takes ~6 s)",
                "clips_per_s": world * 8 / sec5, "ms_per_step": sec5 * 1e3, "steps": args.config5_steps,
                "loss": cfg5_opt["loss"], "launches_per_step": cfg5_opt["launches_per_step"]}
        if cfg5_frozen:
            sec5 = cfg5_frozen["ms"] * 1e-3 / args.config5_steps
            line["config5_frozen"] = {
                "workload": "config 5 with the feature extractors frozen (feature_grad_mult = 0, reference: no_grad): "
                            "training-mode extractor forward, backward of fusion LayerNorm + post_extract_proj + encoder",
                "clips_per_s": world * 8 / sec5, "ms_per_step": sec5 * 1e3, "steps": args.config5_steps,
                "grad_elements": cfg5_frozen["grad_elements"], "loss": cfg5_frozen["loss"],
                "launches_per_step": cfg5_frozen["launches_per_step"]}
        if args.profile_json:
            with open(args.profile_json, "w") as f:
                json.dump({"classes": prof, "total_ms": total_prof_ms}, f, indent=1, sort_keys=True)
        if world == 1 and not args.no_cpu_baseline:
            if full_affinity is not None:
                os.sched_setaffinity(0, full_affinity)      # the CPU arm uses all the host cores it can
            # the oracle is the CHECKER here: same 16 clips, same (bf16-rounded) weights -> CPU time + parity of the
            # benchmarked output
            cores = os.cpu_count() or 1
            import torch.nn.functional as Fnn
            from oracle import avhubert_oracle as ao
            torch.set_num_threads(cores)
            oracle = ao.build_oracle("large", seed=1234, randomize=False)
            sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
            missing = oracle.load_state_dict(sd, strict=False)
            src = {"audio": dev_a[0].float().cpu(), "video": dev_v[0].float().cpu()}
            y_dev = model.extract_finetune({"audio": dev_a[0], "video": dev_v[0]}, None)[0].float().cpu()
            times = []
            with torch.no_grad():
                for i in range(3):
                    t0 = time.perf_counter()
                    y_ref, _ = oracle.extract_finetune(src, None)
                    times.append(time.perf_counter() - t0)
            cos = [float(Fnn.cosine_similarity(y_dev[i].flatten().double(), y_ref[i].flatten().double(), dim=0))
                   for i in range(B_PER_GPU)]
            line["cpu_baseline"] = {
                "value": B_PER_GPU / min(times[1:]), "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"all {B_PER_GPU} clips of one step (the same inputs and weights as the GPU arm), fp32 PyTorch "
                          "CPU oracle (restatement of the reference path), best of 2 after 1 warm-up"}
            line["parity"] = {"vs": "fp32 CPU oracle on the same 16 clips and weights (bf16 gate: cosine >= 0.999 per clip)",
                              "cosine_min_per_clip": min(cos), "cosine_mean": sum(cos) / len(cos),
                              "unexpected_keys": list(missing.unexpected_keys), "missing_keys": list(missing.missing_keys),
                              "logfbank": "parity unpinned (python_speech_features absent; known-answer tests only)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
