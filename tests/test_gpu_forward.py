"""End-to-end parity of AVHubertModel.extract_finetune on a B200 against (a) the golden outputs of the REAL
reference (tests/golden/enc_*.npz) and (b) the fp32 CPU oracle on the same seeded inputs.

Gates (BASELINE.md §5): fp32 mode <= 2e-3 relative (max|y - y_ref| / max|y_ref|), bf16 mode cosine >= 0.999,
padding masks bit-exact.  Dense mode: padded positions are compared too."""
import pytest
import torch

from multimodalvc_b200 import HubertEncoderWrapper

from helpers import cosine, load_encoder_case, make_device_model, rel_err, to_dev

pytestmark = pytest.mark.gpu

FP32_TOL = 2e-3
BF16_COS = 0.999
TINY = ["tiny_av_ragged", "tiny_video_only", "tiny_audio_only", "tiny_layer1", "tiny_postln", "tiny_add"]


def run_case(name, dtype, **cfg_kw):
    c = load_encoder_case(name)
    m = make_device_model(c["oracle"], c["over"], c["size"], dtype, **cfg_kw)
    src, pm = to_dev(c["src"], c["pm"], dtype=dtype)
    y, pm_out = m.extract_finetune(src, pm, output_layer=c["output_layer"])
    torch.cuda.synchronize()
    assert y.dtype == dtype and y.shape == c["y_ref"].shape
    assert torch.isfinite(y).all()
    if pm is not None:
        assert torch.equal(pm_out.cpu(), torch.from_numpy(c["pm_ref"]))
    return y.float().cpu(), c, m


@pytest.mark.parametrize("name", TINY)
def test_fp32_mode_matches_reference_golden_tiny(name):
    y, c, _ = run_case(name, torch.float32)
    assert rel_err(y, c["y_ref"]) < FP32_TOL


@pytest.mark.parametrize("name", TINY)
def test_bf16_mode_matches_reference_golden_tiny(name):
    y, c, _ = run_case(name, torch.bfloat16)
    assert cosine(y, c["y_ref"]) > BF16_COS


def test_fp16_module_like_reference_eval():
    # src/eval.py:155-156,200: model.half(), video cast to fp16
    y, c, _ = run_case("tiny_av_ragged", torch.float16)
    assert cosine(y, c["y_ref"]) > BF16_COS


def test_base_config1_fp32_and_bf16():
    # BASELINE config 1: Base, B=1, T=50
    y, c, _ = run_case("base_b1_t50", torch.float32)
    assert rel_err(y, c["y_ref"]) < FP32_TOL
    y, c, _ = run_case("base_b1_t50", torch.bfloat16)
    assert cosine(y, c["y_ref"]) > BF16_COS


def test_large_ragged_fp32_and_bf16():
    y, c, _ = run_case("large_b2_t40", torch.float32)
    assert rel_err(y, c["y_ref"]) < FP32_TOL
    y, c, _ = run_case("large_b2_t40", torch.bfloat16)
    assert cosine(y, c["y_ref"]) > BF16_COS


def test_stage_level_parity_fp32():
    c = load_encoder_case("tiny_av_ragged")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.float32, capture_stages=True)
    src, pm = to_dev(c["src"], c["pm"])
    m.extract_finetune(src, pm)
    with torch.no_grad():
        stages, _ = c["oracle"].stage_outputs(c["src"], c["pm"])
    B, T = c["pm"].shape
    res = m.read_stage("resnet", B * T * 512).view(B, T, 512).cpu()
    assert rel_err(res, stages["resnet"].transpose(1, 2)) < 1e-3
    fl = m.read_stage("fused_ln", B * T * 256).view(B, T, 256).cpu()
    assert rel_err(fl, stages["fused_ln"]) < 1e-3
    ei = m.read_stage("enc_in", B * T * 128).view(B, T, 128).cpu()
    ref = stages["enc_in"].masked_fill(c["pm"].unsqueeze(-1), 0.0)       # device copy is taken after pad zeroing
    assert rel_err(ei, ref) < 1e-3


def test_stage_level_parity_bf16_frontend_kernels():
    """bf16 mode runs its own frontend kernels (fused stem on TS-MMA, window conv, frame-row convs): check the
    ResEncoder output directly against the fp32 oracle.  Tolerance: 17 convolutions on bf16 activations,
    max-normalised error <= 2e-2 (bf16 has 8 mantissa bits), and cosine >= 0.9995."""
    c = load_encoder_case("tiny_av_ragged")
    with torch.no_grad():
        stages, _ = c["oracle"].stage_outputs(c["src"], c["pm"])
    B, T = c["pm"].shape
    ref = stages["resnet"].transpose(1, 2)
    for chunk in (0, 7):                                   # one launch / several frontend chunks (b0 > 0 paths)
        m = make_device_model(c["oracle"], c["over"], c["size"], torch.bfloat16, capture_stages=True,
                              frontend_chunk_frames=chunk)
        src, pm = to_dev(c["src"], c["pm"], dtype=torch.bfloat16)
        m.extract_finetune(src, pm)
        res = m.read_stage("resnet", B * T * 512).view(B, T, 512).float().cpu()
        assert rel_err(res, ref) < 2e-2 and cosine(res, ref) > 0.9995


@pytest.mark.parametrize("T", [1, 2, 3, 5, 31])
def test_bf16_frontend_short_and_odd_clips(T):
    """The fused stem walks time in frame pairs with a 5-frame ring: clips shorter than the temporal kernel, odd
    lengths (unpaired last frame) and fp32 / fp16 video inputs (generic loader path) against the fp32 oracle."""
    from oracle import avhubert_oracle as ao
    oracle = ao.build_oracle("tiny", seed=77)
    src, _ = ao.synthetic_inputs(2, T, seed=T)
    with torch.no_grad():
        stages, _ = oracle.stage_outputs(src, None)
    ref = stages["resnet"].transpose(1, 2)
    m = make_device_model(oracle, {}, "tiny", torch.bfloat16, capture_stages=True)
    outs = []
    for vdt in (torch.bfloat16, torch.float32, torch.float16):
        s = {"audio": src["audio"].cuda().to(torch.bfloat16), "video": src["video"].cuda().to(vdt)}
        m.extract_finetune(s, None)
        res = m.read_stage("resnet", 2 * T * 512).view(2, T, 512).float().cpu()
        assert torch.isfinite(res).all()
        assert rel_err(res, ref) < 2e-2 and cosine(res, ref) > 0.9995, (T, vdt)
        outs.append(res)


def test_frontend_chunking_is_invisible():
    c = load_encoder_case("tiny_av_ragged")
    src, pm = to_dev(c["src"], c["pm"])
    ys = []
    for chunk in (0, 7, 60):
        m = make_device_model(c["oracle"], c["over"], c["size"], torch.float32, frontend_chunk_frames=chunk)
        ys.append(m.extract_finetune(src, pm)[0].cpu())
    assert torch.equal(ys[0], ys[1]) and torch.equal(ys[0], ys[2])


def test_inputs_are_not_modified_and_views_are_accepted():
    c = load_encoder_case("tiny_av_ragged")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.float32)
    src, pm = to_dev(c["src"], c["pm"])
    assert not src["audio"].is_contiguous()          # collater hands a transposed view
    keep = {k: v.clone() for k, v in src.items()}
    pm_keep = pm.clone()
    y1, _ = m.extract_finetune(src, pm)
    y2, _ = m.extract_finetune({"audio": src["audio"].contiguous(), "video": src["video"]}, pm)
    assert torch.equal(src["audio"], keep["audio"]) and torch.equal(src["video"], keep["video"])
    assert torch.equal(pm, pm_keep)
    assert torch.equal(y1, y2)


def test_wrapper_output_dict_and_layout():
    c = load_encoder_case("tiny_av_ragged")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.float32)
    src, pm = to_dev(c["src"], c["pm"])
    out = HubertEncoderWrapper(m)(source=src, padding_mask=pm)
    assert out["encoder_out"].shape == (c["y_ref"].shape[1], c["y_ref"].shape[0], c["y_ref"].shape[2])
    assert rel_err(out["encoder_out"].transpose(0, 1).cpu(), c["y_ref"]) < FP32_TOL
    assert out["encoder_padding_mask"] is out["padding_mask"]


def test_host_buffer_entry_point_matches_device_call():
    c = load_encoder_case("tiny_av_ragged")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.float32)
    src, pm = to_dev(c["src"], c["pm"])
    y_dev, _ = m.extract_finetune(src, pm)
    y_host = m.extract_finetune_host(c["src"]["video"].contiguous().pin_memory(),
                                     c["src"]["audio"].contiguous().pin_memory(), c["pm"])
    assert torch.equal(y_dev.cpu(), y_host)


def test_reload_after_weight_change_and_dtype_change():
    c = load_encoder_case("tiny_video_only")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.float32)
    src, pm = to_dev(c["src"], c["pm"])
    y0, _ = m.extract_finetune(src, pm)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    sd["encoder.layer_norm.bias"] += 1.0
    m.load_state_dict(sd)
    y1, _ = m.extract_finetune(src, pm)
    assert (y1 - y0 - 1.0).abs().max().item() < 1e-5
    m = m.bfloat16()
    y2, _ = m.extract_finetune({"audio": None, "video": src["video"].bfloat16()}, pm)
    assert y2.dtype == torch.bfloat16 and cosine(y2.float().cpu(), y1.cpu()) > BF16_COS


def test_large_b16_t150_properties():
    """BASELINE config 2 at full size: too slow for the CPU oracle in a test, so size-independent properties:
    (1) batch independence — clip i alone equals clip i inside the batch; (2) zero padding invisibility for
    valid frames; (3) determinism."""
    from oracle import avhubert_oracle as ao
    oracle = ao.build_oracle("large", seed=1234)
    m = make_device_model(oracle, {}, "large", torch.bfloat16)
    src, _ = ao.synthetic_inputs(16, 150, seed=21)
    src, _ = to_dev(src, None, dtype=torch.bfloat16)
    y, _ = m.extract_finetune(src, None)
    y_again, _ = m.extract_finetune(src, None)
    assert torch.equal(y, y_again)
    one = {"audio": src["audio"][3:4], "video": src["video"][3:4]}
    y1, _ = m.extract_finetune(one, None)
    assert cosine(y1.float().cpu(), y[3:4].float().cpu()) > 0.9999
    # pad clip 3 to T=180 with zeros + mask: valid frames unchanged
    v = torch.zeros(1, 1, 180, 88, 88, device="cuda", dtype=torch.bfloat16)
    v[:, :, :150] = one["video"]
    a = torch.zeros(1, 104, 180, device="cuda", dtype=torch.bfloat16)
    a[:, :, :150] = one["audio"]
    pm = torch.zeros(1, 180, dtype=torch.bool, device="cuda")
    pm[:, 150:] = True
    yp, _ = m.extract_finetune({"audio": a, "video": v}, pm)
    assert cosine(yp[:, :150].float().cpu(), y1.float().cpu()) > 0.9995


def test_extract_features_matches_reference_golden():
    """AVHubertModel.extract_features (hubert.py:676-692): conv features (encoder input with padded frames zeroed),
    layer-k features and the full output against outputs of the REAL reference (enc_extract_features.npz)."""
    import numpy as np
    import os
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "enc_extract_features.npz"))
    c = load_encoder_case("tiny_av_ragged")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.float32)
    src, pm = to_dev(c["src"], c["pm"])
    for key, kw in {"conv": dict(ret_conv=True), "layer1": dict(output_layer=1), "full": dict()}.items():
        y, pm_out = m.extract_features(src, pm, mask=False, **kw)
        assert rel_err(y.cpu(), torch.from_numpy(z[key])) < FP32_TOL, key
        assert torch.equal(pm_out.cpu(), torch.from_numpy(z["pm_out"]))
    y, _ = m.extract_features(src, pm, ret_conv=True)
    assert not y[c["pm"].cuda()].any()                       # padded frames of the conv features are zero
    with pytest.raises(ValueError):
        m.extract_features({"audio": None, "video": src["video"]}, pm)
    mb = make_device_model(c["oracle"], c["over"], c["size"], torch.bfloat16)
    srcb, _ = to_dev(c["src"], c["pm"], dtype=torch.bfloat16)
    yb, _ = mb.extract_features(srcb, pm, ret_conv=True)
    assert cosine(yb.float().cpu(), torch.from_numpy(z["conv"])) > BF16_COS


def test_hubert_encoder_ctc_head():
    """HubertEncoder (hubert_asr.py:251-354): T x B x C output, three-key dict, optional vocabulary projection."""
    from multimodalvc_b200 import HubertEncoder
    c = load_encoder_case("tiny_av_ragged")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.bfloat16)
    src, pm = to_dev(c["src"], c["pm"], dtype=torch.bfloat16)
    enc = HubertEncoder(m).cuda().eval()
    out = enc(src, pm)
    y, _ = m.extract_finetune(src, pm)
    assert set(out) == {"encoder_out", "encoder_padding_mask", "padding_mask"}
    assert torch.equal(out["encoder_out"], y.transpose(0, 1)) and torch.equal(out["padding_mask"], pm)
    assert torch.equal(enc(src, pm, tbc=False)["encoder_out"], y)
    head = HubertEncoder(m, tgt_dict_size=41).cuda().to(torch.bfloat16).eval()          # CTC vocabulary of 41 units
    torch.nn.init.normal_(head.proj.bias, std=0.5)
    o = head(src, pm)["encoder_out"]
    assert o.shape == (y.size(1), y.size(0), 41)
    ref = (y.float() @ head.proj.weight.float().t() + head.proj.bias.float()).transpose(0, 1)
    assert (o.float() - ref).abs().max().item() < 3e-2 * ref.abs().max().item() + 1e-2   # bf16 output rounding
    with pytest.raises(RuntimeError):
        head.train()(src, pm)


def test_cuda_graph_replay_matches_direct_launches():
    """The plan-internal runs of the launch list are captured into CUDA graphs on the second call of a shape and
    replayed afterwards WHATEVER tensors the caller passes (the steps that read caller pointers stay direct launches).
    Replays with fresh input tensors, calls on another stream must reproduce the direct results bit for bit, and must
    read the CURRENT contents of the buffers."""
    c = load_encoder_case("tiny_av_ragged")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.bfloat16)
    src, pm = to_dev(c["src"], c["pm"], dtype=torch.bfloat16)
    y0 = m.extract_finetune(src, pm)[0].clone()                  # direct
    outs = [m.extract_finetune(src, pm)[0].clone() for _ in range(3)]          # capture, replay, replay (fresh outputs)
    assert all(torch.equal(y0, y) for y in outs)
    src2 = {k: v.clone() for k, v in src.items()}                # same values at new addresses
    assert torch.equal(m.extract_finetune(src2, pm.clone())[0], y0)
    # same addresses, new contents: the graph must see them
    src2["video"].mul_(0.5)
    y_half = m.extract_finetune(src2, pm)[0].clone()
    assert not torch.equal(y_half, y0)
    src3 = {"audio": src["audio"], "video": src["video"] * 0.5}
    assert torch.equal(m.extract_finetune(src3, pm)[0], y_half)
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    from multimodalvc_b200 import _lib
    with torch.cuda.stream(st):
        ys = [m.extract_finetune(src, pm)[0] for _ in range(3)]
        g0 = _lib.load().avh_graph_launch_count()
        fresh = {k: v.clone() for k, v in src.items()}           # new addresses on a capturable stream: still a replay
        ys.append(m.extract_finetune(fresh, pm.clone())[0])
        assert _lib.load().avh_graph_launch_count() >= g0 + 2    # graph segments, not ~200 direct launches
    st.synchronize()
    assert all(torch.equal(y0, y) for y in ys)


def test_forward_inside_a_user_cuda_graph():
    """A caller may capture extract_finetune into its own CUDA graph (static input/output tensors): the library then
    records plain launches into that capture instead of starting a nested one."""
    c = load_encoder_case("tiny_av_ragged")
    m = make_device_model(c["oracle"], c["over"], c["size"], torch.bfloat16)
    src, pm = to_dev(c["src"], c["pm"], dtype=torch.bfloat16)
    y_ref = m.extract_finetune(src, pm)[0].clone()
    static_src = {k: v.clone() for k, v in src.items()}
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):                       # plan for this stream + kernel configuration before capture
        m.extract_finetune(static_src, pm)
    torch.cuda.current_stream().wait_stream(st)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        y_static = m.extract_finetune(static_src, pm)[0]
    static_src["video"].copy_(src["video"] * 0.5)
    g.replay()
    torch.cuda.synchronize()
    y_half = m.extract_finetune({"audio": src["audio"], "video": src["video"] * 0.5}, pm)[0]
    assert torch.equal(y_static, y_half)
    static_src["video"].copy_(src["video"])
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(y_static, y_ref)


def test_many_shapes_plan_eviction_and_graph_reuse():
    """More distinct (B, T) shapes than the plan cache holds (8): plans and their CUDA graphs are evicted and rebuilt
    while earlier work may still be queued; every shape must reproduce its first result bit for bit afterwards."""
    from oracle import avhubert_oracle as ao
    oracle = ao.build_oracle("tiny", seed=1234)
    m = make_device_model(oracle, {}, "tiny", torch.bfloat16)
    shapes = [(1, 3), (2, 5), (1, 8), (3, 4), (2, 9), (1, 12), (2, 2), (3, 7), (1, 17), (2, 11), (4, 3)]
    inputs, first = [], []
    for i, (B, T) in enumerate(shapes):
        src, _ = ao.synthetic_inputs(B, T, seed=100 + i)
        src = {k: v.cuda().to(torch.bfloat16) for k, v in src.items()}
        inputs.append(src)
        first.append(m.extract_finetune(src, None)[0].clone())
    for rnd in range(3):
        for src, y0 in zip(inputs, first):
            assert torch.equal(m.extract_finetune(src, None)[0], y0)
    torch.cuda.synchronize()
