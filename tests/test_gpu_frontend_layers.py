"""Lip-frontend kernels layer by layer against a float64 reference.

Every intermediate map of the video ResNet (the stages 'stem', 'layer{L}.{b}.mid', 'layer{L}.{b}.out',
'layer{L}.0.ds' and 'resnet', see AVHubertModel.read_stage) is compared element by element with a float64
computation of that one layer from the device's own input map: the previous stage read back exactly (bf16 values are
exact in fp32), or for the stem the video the kernel read.  Weights go through the packer's rounding: bf16(w) for the
stem and plain convolutions, bf16(s2 w2) and bf16(s_ds w_ds) with the summed bias for the bf16 eval path's conv2 with
the shortcut folded into the same GEMM; BatchNorm scale and bias as the packer computes them in fp32 from the values
the module holds (bf16 statistics for a bf16 module).

Gates: bf16 maps |y - ref| <= 2^-8 |ref| + 1e-4 max|ref| on every element (one output rounding, plus fp32
accumulation order); fp32 mode one max|y - ref| / max|ref| bound per map; the shared zero row and column of every
padded map exactly 0.0, because the next convolution reads them as padding.  The forward has no kinks that rounding
could move across (PReLU and max-pool are continuous, bf16 rounding commutes with max), so these gates are strict."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import avhubert_oracle as ao
from oracle import video_oracle as vo

from helpers import cosine, make_device_model, rel_err

pytestmark = pytest.mark.gpu

R = "feature_extractor_video.resnet."
HS = [22, 11, 6, 3]                      # image size of the stem output and of layers 1-4
BF16_REL, BF16_ABS = 2.0 ** -8, 1e-4
# fp32 mode (three bf16 split products per GEMM): the worst map measured on a B200 (1000 W power limit) over the fp32
# cases below was 1.34e-5 (layer2.0.mid of the multi-chunk case); the other maps measured 6.98e-8 to 1.19e-5
FP32_REL = 5e-5


@pytest.fixture(scope="module")
def oracle():
    return ao.build_oracle("tiny", seed=1234)


class Ref:
    """float64 reference of the frontend's layers with the packer's weights (api.cu pack_conv / pack_all), computed from
    the parameters and buffers the device model holds: a bf16 module hands bf16 BatchNorm statistics, affine parameters
    and PReLU slopes to the packer, which computes in fp32 from those values."""

    def __init__(self, model, bf16):
        self.sd = {k[len(R):]: v.detach().float().cpu() for k, v in model.state_dict().items() if k.startswith(R)}
        self.bf16 = bf16

    def fold(self, bn):                  # 1/sqrt(var + 1e-5f) in fp32, like the packer
        g, b, m, v = (self.sd[bn + s] for s in (".weight", ".bias", ".running_mean", ".running_var"))
        sc = g * (1.0 / torch.sqrt(v + 1e-5))
        return sc, b - m * sc

    def w(self, key, scale=None):
        w = self.sd[key]
        if scale is not None:            # BN scale folded into the weights, in fp32
            w = w * scale.view(-1, *[1] * (w.dim() - 1))
        return w.to(torch.bfloat16).double() if self.bf16 else w.double()

    def prelu(self, x, key):
        s = self.sd[key].double().view(1, -1, *[1] * (x.dim() - 2))
        return torch.where(x > 0, x, x * s)

    @staticmethod
    def affine(x, sc, bi):
        shape = (1, -1) + (1,) * (x.dim() - 2)
        return x * sc.double().view(shape) + bi.double().view(shape)

    def stem(self, clip, t0, t1):
        """Frames [t0, t1) of one clip [1, 1, Tc, 88, 88] -> [t1 - t0, 64, 22, 22].  Input frames outside [t0 - 2, t1 + 2)
        do not reach them, so only that window is convolved (zero temporal padding at the clip's own ends)."""
        lo, hi = max(0, t0 - 2), min(clip.shape[2], t1 + 2)
        y = F.conv3d(clip[:, :, lo:hi].double(), self.w("frontend3D.0.weight"), stride=(1, 2, 2), padding=(2, 3, 3))
        y = self.prelu(self.affine(y, *self.fold("frontend3D.1")), "frontend3D.2.weight")
        y = F.max_pool3d(y, (1, 3, 3), (1, 2, 2), (0, 1, 1))         # pads with -inf
        return y[0, :, t0 - lo:t1 - lo].transpose(0, 1)

    def mid(self, L, b, x):
        pre = f"trunk.layer{L}.{b}."
        y = F.conv2d(x, self.w(pre + "conv1.weight"), stride=2 if (L > 1 and b == 0) else 1, padding=1)
        return self.prelu(self.affine(y, *self.fold(pre + "bn1")), pre + "relu1.weight")

    def ds(self, L, x):
        pre = f"trunk.layer{L}.0."
        return self.affine(F.conv2d(x, self.w(pre + "downsample.0.weight"), stride=2), *self.fold(pre + "downsample.1"))

    def out(self, L, b, mid, x, ds=None):
        """Block output from the device's conv1 output `mid`, block input `x` and, where the device writes one, its
        downsample map `ds`.  Block 0 of layers 2-4 without a downsample map: the bf16 eval path's single GEMM."""
        pre = f"trunk.layer{L}.{b}."
        s2, b2 = self.fold(pre + "bn2")
        if L > 1 and b == 0 and ds is None:
            sd, bd = self.fold(pre + "downsample.1")
            y = (F.conv2d(mid, self.w(pre + "conv2.weight", s2), padding=1) +
                 F.conv2d(x, self.w(pre + "downsample.0.weight", sd), stride=2) + (b2 + bd).double().view(1, -1, 1, 1))
        else:
            y = self.affine(F.conv2d(mid, self.w(pre + "conv2.weight"), padding=1), s2, b2) + (x if ds is None else ds)
        return self.prelu(y, pre + "relu2.weight")


class Stages:
    """Reads the frontend stages of the model's last forward; `nf` frames (the last frontend chunk)."""

    def __init__(self, m, nf, fp32, case):
        self.m, self.nf, self.fp32, self.case = m, nf, fp32, case
        self.errs = {}

    def padded(self, L):                 # stem and layer 1 always; every layer in fp32 mode
        return L <= 1 or self.fp32

    def read(self, name, L):
        """Device map of stage `name` as [nf, H, H, C] on the device; checks the pad ring of a padded layout."""
        H, C = HS[max(L, 1) - 1], 64 << max(L - 1, 0)
        S = H + 1 if self.padded(L) else H
        t = self.m.read_stage(name, self.nf * S * S * C).view(self.nf, S, S, C)
        if S > H:
            assert not t[:, H].any() and not t[:, :, H].any(), f"{self.case}: {name}: pad row/column not zero"
        return t[:, :H, :H]

    @staticmethod
    def frames(t, idx):                  # [n, C, H, W] float64 on the CPU
        return t[idx.to(t.device)].permute(0, 3, 1, 2).double().cpu()

    def check(self, name, y, ref):
        if self.fp32:
            e = rel_err(y, ref)
            self.errs[name] = e
            assert e <= FP32_REL, f"{self.case}: {name}: max|y - ref| / max|ref| = {e:.3e}"
            return
        err = (y - ref).abs()
        bad = err > BF16_REL * ref.abs() + BF16_ABS * ref.abs().max()
        if bad.any():
            i = int(bad.flatten().nonzero()[0])
            pos = np.unravel_index(i, tuple(y.shape))
            raise AssertionError(f"{self.case}: {name}: {int(bad.sum())} of {bad.numel()} elements outside the bf16 gate; "
                                 f"first at (frame, c, y, x) = {pos}: device {y.flatten()[i]:.6g}, reference "
                                 f"{ref.flatten()[i]:.6g}, max|ref| {ref.abs().max():.4g}")

    def check_stem(self, ref, clips):
        """clips: (clip video [1, 1, Tc, 88, 88] as the kernel read it, first frame of the clip in the stage, t0, t1)."""
        stem = self.read("stem", 0)
        for video, f0, t0, t1 in clips:
            idx = torch.arange(f0 + t0, f0 + t1)
            self.check(f"stem[frames {f0 + t0}..{f0 + t1 - 1}]", self.frames(stem, idx), ref.stem(video, t0, t1))

    def check_trunk(self, ref, idx, resnet_row0):
        """Every trunk stage at chunk-local frames idx, each from the device's input map; then 'resnet' (rows of the
        chunk start at resnet_row0) against the float64 mean of layer4.1.out."""
        x = self.frames(self.read("stem", 0), idx)
        for L in range(1, 5):
            for b in range(2):
                nm = f"layer{L}.{b}"
                mid = self.frames(self.read(nm + ".mid", L), idx)
                self.check(nm + ".mid", mid, ref.mid(L, b, x))
                ds = None
                if L > 1 and b == 0 and self.fp32:
                    ds = self.frames(self.read(nm + ".ds", L), idx)
                    self.check(nm + ".ds", ds, ref.ds(L, x))
                out = self.frames(self.read(nm + ".out", L), idx)
                self.check(nm + ".out", out, ref.out(L, b, mid, x, ds))
                x = out
        res = self.m.read_stage("resnet", (resnet_row0 + self.nf) * 512).view(-1, 512)[resnet_row0:]
        self.check("resnet", res[idx.to(res.device)].double().cpu(), x.mean(dim=(2, 3)))


def pick_frames(nf, clip_starts, extra, n_random, seed=0):
    """Chunk-local trunk frames: first and last frame of every clip, 128-frame tile edges, `extra`, and a few random
    frames in every 128-frame tile."""
    s = {0, nf - 1} | {f for f in extra if 0 <= f < nf}
    for a, b in zip(clip_starts, list(clip_starts[1:]) + [nf]):
        s |= {a, b - 1}
    s |= {f for k in range(128, nf, 128) for f in (k - 1, k)}
    g = torch.Generator().manual_seed(seed)
    for k in range(0, nf, 128):
        n = min(128, nf - k)
        s |= {k + int(i) for i in torch.randint(0, n, (n_random,), generator=g)}
    return torch.tensor(sorted(s))


def last_chunk(B, T, chunk_frames):
    """First clip and clip count of the last frontend chunk (build_plan: whole clips, ceil(B / CB) chunks split evenly)."""
    cb = max(1, (chunk_frames if chunk_frames > 0 else 2400) // T)
    n = (B + cb - 1) // cb
    cb = (B + n - 1) // n
    b0 = (B - 1) // cb * cb
    return b0, B - b0


def video_input(B, T, seed, dtype):
    src, _ = ao.synthetic_inputs(B, T, seed=seed, audio=False)
    return src["video"].to(dtype)


def run_dense(oracle, dtype, B, T, chunk=0, stem_clips=None, trunk_frames=None, case=""):
    """Video-only eval forward on a dense [B, T] batch, then every stage of the last frontend chunk."""
    fp32 = dtype == torch.float32
    m = make_device_model(oracle, {}, "tiny", dtype, capture_stages=True, frontend_chunk_frames=chunk)
    v = video_input(B, T, seed=B * 1000 + T, dtype=dtype)
    m.extract_finetune({"audio": None, "video": v.cuda()}, None)
    torch.cuda.synchronize()
    b0, nb = last_chunk(B, T, chunk)
    st = Stages(m, nb * T, fp32, case)
    ref = Ref(m, bf16=not fp32)
    clips = range(nb) if stem_clips is None else stem_clips
    st.check_stem(ref, [(v[b0 + c:b0 + c + 1], c * T, 0, T) for c in clips])
    idx = trunk_frames if trunk_frames is not None else torch.arange(nb * T)
    st.check_trunk(ref, idx, b0 * T)
    return st


# ---------------------------------------------------------------------------------------------------------- bf16 eval
@pytest.mark.parametrize("B,T,edge", [
    (1, 1, "one frame: an unpaired stem frame, a single partial tile everywhere"),
    (2, 3, "clips shorter than the stem's 5-frame temporal kernel"),
    (3, 43, "129 frames: one frame past a 128-frame tile, odd T"),
    (2, 128, "exactly one 256-frame CTA-pair tile in layers 3-4"),
    (1, 257, "one frame past a 256-frame CTA-pair tile"),
])
def test_bf16_layers_dense(oracle, B, T, edge):
    nf = B * T
    idx = None if nf <= 48 else pick_frames(nf, [c * T for c in range(B)], [255, 256], 6)
    run_dense(oracle, torch.bfloat16, B, T, trunk_frames=idx, case=f"bf16 B={B} T={T} ({edge})")


def test_bf16_layers_config2_chunk(oracle):
    """The benchmark's 2400-frame chunk (16 x 150): the stem on the first, a middle and the last clip, the trunk on
    ~100 frames including every 128-frame tile edge and the ends of those clips."""
    B, T = 16, 150
    extra = [0, 127, 128, 255, 256, 2399] + [c * T + d for c in (0, 8, 15) for d in (0, T - 1)]
    idx = pick_frames(B * T, [c * T for c in range(B)], extra, 2)
    run_dense(oracle, torch.bfloat16, B, T, stem_clips=[0, 8, 15], trunk_frames=idx, case="bf16 config-2 chunk")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_layers_last_of_several_chunks(oracle, dtype):
    """B = 5, T = 60 in 128-frame chunks: chunks of 2, 2 and 1 clips; the stages hold the last, one-clip chunk."""
    assert last_chunk(5, 60, 128) == (4, 1)
    st = run_dense(oracle, dtype, 5, 60, chunk=128, case=f"{dtype} multi-chunk")
    if st.fp32:
        print("fp32 multi-chunk max rel err per map:", {k: f"{v:.2e}" for k, v in st.errs.items()})


def test_bf16_layers_packed_ragged(oracle):
    """cfg.ragged = 'packed': clips back to back in one chunk (the stem's ragged work list, frames of different clips
    in one tile); every clip's stem referenced on its own."""
    lengths = [1, 2, 5, 150, 37, 600, 129]
    B, T = len(lengths), max(lengths)
    src, pm = ao.synthetic_inputs(B, T, lengths=lengths, seed=5, audio=False)
    v = src["video"].to(torch.bfloat16)
    m = make_device_model(oracle, {}, "tiny", torch.bfloat16, capture_stages=True, ragged="packed")
    m.extract_finetune({"audio": None, "video": v.cuda()}, pm.cuda(), lengths=lengths)
    torch.cuda.synchronize()
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]).tolist()
    nf = sum(lengths)
    st = Stages(m, (nf + 127) // 128 * 128, False, "bf16 packed ragged")     # the plan's 128-frame bucket
    ref = Ref(m, bf16=True)
    st.check_stem(ref, [(v[c:c + 1, :, :n], starts[c], 0, n) for c, n in enumerate(lengths)])
    st.check_trunk(ref, pick_frames(nf, starts, [], 4), 0)


@pytest.mark.parametrize("vdt", ["bf16", "fp32", "fp16", "uint8"])
def test_bf16_stem_video_dtypes(oracle, vdt):
    """The fused stem's loaders: bf16 video (16-byte fast path), fp32 / fp16 (generic path, rounded to bf16 on load)
    and raw uint8 frames, normalised on the device into bf16 (pinned by tests/test_gpu_video.py)."""
    B, T = 2, 7
    m = make_device_model(oracle, {}, "tiny", torch.bfloat16, capture_stages=True)
    if vdt == "uint8":
        frames = vo.synthetic_frames(B * T, 96, 96, seed=3)
        dev = torch.from_numpy(frames).view(B, 1, T, 96, 96)
        read = torch.from_numpy(vo.video_transform(frames).astype(np.float32)).to(torch.bfloat16).view(B, 1, T, 88, 88)
    else:
        dt = {"bf16": torch.bfloat16, "fp32": torch.float32, "fp16": torch.float16}[vdt]
        dev = video_input(B, T, seed=31, dtype=dt)
        read = dev.to(torch.bfloat16)             # the kernel rounds fp32 / fp16 pixels to bf16
    m.extract_finetune({"audio": None, "video": dev.cuda()}, None)
    torch.cuda.synchronize()
    st = Stages(m, B * T, False, f"bf16 stem, {vdt} video")
    st.check_stem(Ref(m, bf16=True), [(read[c:c + 1], c * T, 0, T) for c in range(B)])


# ---------------------------------------------------------------------------------------------------------- fp32 mode
@pytest.mark.parametrize("B,T", [(2, 37), (1, 1)])
def test_fp32_layers(oracle, B, T):
    st = run_dense(oracle, torch.float32, B, T, case=f"fp32 B={B} T={T}")
    print(f"fp32 B={B} T={T} max rel err per map:", {k: f"{v:.2e}" for k, v in st.errs.items()})


# ------------------------------------------------------------------------------- training-mode forward over chunks
def bn_flat(mods):
    return torch.cat([torch.cat([b.running_mean.float().cpu(), b.running_var.float().cpu()]) for b in mods])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("chunk", [0, 7])
def test_train_mode_forward_batch_statistics_over_chunks(dtype, chunk):
    """model.train() under no_grad normalises with the statistics of the WHOLE batch and updates the running statistics
    once, as nn.BatchNorm does, whatever frontend_chunk_frames is (7 with T = 20 would be three one-clip chunks)."""
    from oracle.make_golden_train import bn_modules
    B, T = 3, 20
    oracle = ao.build_oracle("tiny", seed=1234)
    m = make_device_model(oracle, {}, "tiny", dtype, frontend_chunk_frames=chunk, dropout=0.0, attention_dropout=0.0,
                          activation_dropout=0.0, dropout_input=0.0, encoder_layerdrop=0.0)
    src, _ = ao.synthetic_inputs(B, T, seed=23, audio=False)
    m.train()
    with torch.no_grad():
        y, _ = m.extract_finetune({"audio": None, "video": src["video"].to("cuda", dtype)}, None)
        oracle.train()
        y_ref, _ = oracle.extract_finetune({"audio": None, "video": src["video"]}, None)
    y = y.float().cpu()
    bn, bn_ref = bn_flat(m._bn_modules()), bn_flat(bn_modules(oracle))
    if dtype == torch.float32:
        assert rel_err(y, y_ref) < 2e-3
        assert (bn - bn_ref).abs().max() < 1e-4 * bn_ref.abs().max()
    else:
        assert cosine(y, y_ref) > 0.999
        assert (bn - bn_ref).abs().max() < 2e-2 * bn_ref.abs().max()       # bf16 buffers, bf16 conv outputs
