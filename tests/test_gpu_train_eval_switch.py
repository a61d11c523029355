"""Switching one model between training and evaluation without a re-pack through the host.

After training steps (optimizer updates, training-mode BatchNorm moving the running statistics) the first eval forward
refreshes the packed weights in place on the device (avh_refresh_eval_weights_device): the training forms from the
parameters, the eval-only forms (BatchNorm folds, the conv2 + shortcut GEMM weights) from the parameters and the
BatchNorm buffers.  The refresh computes what the host packers compute, so every comparison here is bit for bit
(torch.equal) against a fresh model that loaded the same state dict through the host.  The handle, its plans and its
captured graphs survive the switch: avh_finalize_weights is never called again, and the training plan is reused."""
import contextlib
import ctypes
import re
import shutil
import subprocess
from types import SimpleNamespace

import pytest
import torch

from oracle import avhubert_oracle as ao

B, T = 2, 18
STAGE_CAP = B * T * 23 * 23 * 64          # the largest stage of the tiny model (stem and layer 1 maps, padded)


@pytest.fixture
def finalize_spy(monkeypatch):
    """Handles avh_finalize_weights is called with (it drops every plan, arena and captured graph)."""
    from multimodalvc_b200 import _lib
    lib = _lib.load()
    real = lib.avh_finalize_weights
    calls = []

    def spy(h):
        calls.append(h.value if isinstance(h, ctypes.c_void_p) else h)
        return real(h)

    monkeypatch.setattr(lib, "avh_finalize_weights", spy)
    return calls


def plan_count(handle):
    from multimodalvc_b200 import _lib
    n = ctypes.c_int32()
    _lib.check(_lib.load().avh_plan_count(handle, ctypes.byref(n)))
    return n.value


def stage(m, name):
    """A stage of m's last forward, zero beyond what the library writes (its element count differs per mode)."""
    from multimodalvc_b200 import _lib
    dst = torch.zeros(STAGE_CAP, device="cuda", dtype=torch.float32)
    _lib.check(_lib.load().avh_read_stage(m._handle, name.encode(), ctypes.c_void_p(dst.data_ptr()), STAGE_CAP,
                                          ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return dst


def stage_names(fp32):
    names = ["stem", "resnet", "fused", "fused_ln", "enc_in"]
    for L in range(1, 5):
        for b in range(2):
            names += [f"layer{L}.{b}.mid", f"layer{L}.{b}.out"]
        if fp32 and L > 1:
            names.append(f"layer{L}.0.ds")         # the bf16 eval path folds the shortcut into conv2's GEMM
    return names


def make_model(cfg, sd, dtype):
    from multimodalvc_b200 import AVHubertModel
    m = AVHubertModel(cfg)
    m.remove_pretraining_modules()
    m.load_state_dict(sd, strict=False)
    return m.to(device="cuda", dtype=dtype)


def side(stream):
    return torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()


def cycles():
    """Default stream, then twice a side stream: there the refresh runs as a captured graph, replayed the second time
    with the new parameter and statistics values."""
    s = torch.cuda.Stream()
    return [None, s, s]


def check_eval(m, cfg, dtype, dsrc, pm, handle, fp32):
    """m's eval forward equals a fresh model's, stage by stage; returns the fresh model."""
    m.eval()
    with torch.no_grad():
        e, _ = m.extract_finetune(dsrc, pm)
    assert m._handle is handle and not m._dirty
    stages = {n: stage(m, n) for n in stage_names(fp32)}
    fresh = make_model(cfg, m.state_dict(), dtype).eval()
    with torch.no_grad():
        e2, _ = fresh.extract_finetune(dsrc, pm)
    assert torch.equal(e, e2)
    for n, v in stages.items():
        assert torch.equal(v, stage(fresh, n)), n
    return fresh


def check_buffers(m, fresh):
    fb = dict(fresh.named_buffers())
    for n, b in m.named_buffers():
        assert torch.equal(b, fb[n]), n


def _train_cfg(fgm, compute, fuse):
    from multimodalvc_b200 import AVHubertConfig
    return AVHubertConfig.named("tiny", modality_fuse=fuse, feature_grad_mult=fgm, trainable=True, compute_dtype=compute,
                                capture_stages=True, dropout=0.0, attention_dropout=0.0, activation_dropout=0.0,
                                encoder_layerdrop=0.0, dropout_input=0.0)


def _switch_trainable(fgm, compute, fuse, finalize_spy):
    o = ao.build_oracle("tiny", seed=1234, modality_fuse=fuse)
    src, pm = ao.synthetic_inputs(B, T, lengths=[18, 13], seed=29)
    cfg = _train_cfg(fgm, compute, fuse)
    m = make_model(cfg, o.state_dict(), torch.float32).train()
    dsrc, dpm = {k: v.cuda() for k, v in src.items()}, pm.cuda()
    opt = torch.optim.SGD(m.parameters(), lr=0.05, momentum=0.9)

    def step():
        opt.zero_grad()
        y, _ = m.extract_finetune(dsrc, dpm)
        (y[~dpm] ** 2).mean().backward()
        opt.step()
        return y.detach()

    handle = None
    for stream in cycles():
        if stream is not None:
            stream.wait_stream(torch.cuda.current_stream())
        with side(stream):
            step(); step()
            if handle is None:
                handle = m._handle
                finalize_spy.clear()          # the first step packed the weights; nothing may re-pack them from here on
            fresh = check_eval(m, cfg, torch.float32, dsrc, dpm, handle, compute == "fp32")
            n_plans = plan_count(handle)
            assert n_plans >= 2                             # the eval plan joins the training plans: none dropped
            # back to training: the next step equals the fresh model's first one, and so do the statistics it leaves
            m.train(); fresh.train()
            y = step()
            y2, _ = fresh.extract_finetune(dsrc, dpm)
            assert torch.equal(y, y2.detach())
            check_buffers(m, fresh)
            assert m._handle is handle and plan_count(handle) == n_plans          # the training plan was reused
            del fresh
        if stream is not None:
            torch.cuda.current_stream().wait_stream(stream)
    assert handle.value not in finalize_spy


@pytest.mark.gpu
@pytest.mark.parametrize("fuse", ["concat", "add"])
@pytest.mark.parametrize("compute", ["bf16", "fp32"])
def test_whole_model_train_eval_switch(compute, fuse, finalize_spy):
    """feature_grad_mult = 1: every parameter trains, the training-mode BatchNorm moves the running statistics."""
    _switch_trainable(1.0, compute, fuse, finalize_spy)


@pytest.mark.gpu
@pytest.mark.parametrize("compute", ["bf16", "fp32"])
def test_frozen_extractors_train_eval_switch(compute, finalize_spy):
    """feature_grad_mult = 0: the extractors run under no_grad in training mode (statistics move, weights do not)."""
    _switch_trainable(0.0, compute, "concat", finalize_spy)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_frozen_encoder_in_train_mode_switch(dtype, finalize_spy):
    """MMS-LLaMA's form: a model that is not trainable runs in .train() under no_grad, so only the BatchNorm running
    statistics move — a bf16 module holds them rounded to bf16, and the eval folds must start from those values."""
    from multimodalvc_b200 import AVHubertConfig
    o = ao.build_oracle("tiny", seed=1234)
    src, pm = ao.synthetic_inputs(B, T, lengths=[18, 13], seed=31)
    cfg = AVHubertConfig.named("tiny", capture_stages=True, dropout=0.0, attention_dropout=0.0, activation_dropout=0.0,
                               encoder_layerdrop=0.0, dropout_input=0.0)
    m = make_model(cfg, o.state_dict(), dtype).train()
    dsrc = {k: v.cuda().to(dtype) for k, v in src.items()}
    dpm = pm.cuda()
    handle = None
    for stream in cycles():
        if stream is not None:
            stream.wait_stream(torch.cuda.current_stream())
        with side(stream), torch.no_grad():
            for _ in range(2):
                m.extract_finetune(dsrc, dpm)
            if handle is None:
                handle = m._handle
                finalize_spy.clear()
            fresh = check_eval(m, cfg, dtype, dsrc, dpm, handle, dtype == torch.float32)
            n_plans = plan_count(handle)
            assert n_plans >= 2
            m.train(); fresh.train()
            y, _ = m.extract_finetune(dsrc, dpm)
            y2, _ = fresh.extract_finetune(dsrc, dpm)
            assert torch.equal(y, y2)
            check_buffers(m, fresh)
            assert m._handle is handle and plan_count(handle) == n_plans
            del fresh
        if stream is not None:
            torch.cuda.current_stream().wait_stream(stream)
    assert handle.value not in finalize_spy


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_bare_encoder_train_eval_switch(dtype, finalize_spy):
    """TransformerEncoder(trainable=True): no eval-only forms; the eval forward picks up the optimizer steps since the
    last training forward on the device."""
    from multimodalvc_b200.sr_predictor import TransformerEncoder
    args = SimpleNamespace(encoder_embed_dim=128, encoder_ffn_embed_dim=256, encoder_attention_heads=2, encoder_layers=2,
                           conv_pos=128, conv_pos_groups=16, layer_norm_first=True, dropout=0.0, attention_dropout=0.0,
                           activation_dropout=0.0, encoder_layerdrop=0.0)
    torch.manual_seed(5)
    enc = TransformerEncoder(args, trainable=True).to(device="cuda", dtype=dtype).train()
    g = torch.Generator().manual_seed(8)
    x = torch.randn(B, T, 128, generator=g).to(device="cuda", dtype=dtype)
    pm = torch.zeros(B, T, dtype=torch.bool)
    pm[1, 13:] = True
    pm = pm.cuda()
    opt = torch.optim.SGD(enc.parameters(), lr=0.05, momentum=0.9)

    def step(mod):
        opt.zero_grad()
        y, _ = mod(x, pm)
        (y[~pm].float() ** 2).mean().backward()
        opt.step()
        return y.detach()

    handle = None
    for stream in cycles():
        if stream is not None:
            stream.wait_stream(torch.cuda.current_stream())
        with side(stream):
            for _ in range(3):
                step(enc)
            if handle is None:
                handle = enc._handle
                finalize_spy.clear()
            enc.eval()
            with torch.no_grad():
                e, _ = enc(x, pm)
            assert enc._handle is handle and not enc._dirty
            fresh = TransformerEncoder(args, trainable=True)
            fresh.load_state_dict(enc.state_dict())
            fresh = fresh.to(device="cuda", dtype=dtype).eval()
            with torch.no_grad():
                e2, _ = fresh(x, pm)
            assert torch.equal(e, e2)
            n_plans = plan_count(handle)
            assert n_plans >= 2
            enc.train()
            step(enc)
            assert enc._handle is handle and plan_count(handle) == n_plans
            del fresh
        if stream is not None:
            torch.cuda.current_stream().wait_stream(stream)
    assert handle.value not in finalize_spy


def test_host_packers_have_no_fma():
    """The host packers fold BatchNorm with separately rounded fp32 operations, as the device refresh kernels do: a
    fused multiply-add in the host code would break their bit-identity."""
    objdump = shutil.which("objdump")
    if objdump is None:
        pytest.skip("objdump not available")
    from multimodalvc_b200 import build
    lib = build.build()
    asm = subprocess.run([objdump, "-d", lib], capture_output=True, text=True, check=True).stdout
    fma = re.findall(r"\s(v?f(?:n)?m(?:add|sub)\w*|fml[as])\s", asm)
    assert not fma, sorted(set(fma))[:10]
