"""The device training step with post-LN layers (layer_norm_first=False: wav2vec2.py:872-879 and :993-1012, the
LayerNorm after the positional conv, no final LayerNorm) for the bare TransformerEncoder, the frozen-extractor tail and
the whole model, with dropout, activation dropout, dropout_input and LayerDrop.

The reference is float64 torch.autograd on the oracle's post-LN modules (pinned against the real AVHubertModel by the
tiny_postln golden), restated with the library's masks injected at each site: every mask is rebuilt exactly with
avh_dropout (same seed, same site id) on a tensor of ones — site 1 dropout_input, 2 after the encoder LayerNorm,
16+4l / 17+4l / 18+4l dropout1 / activation dropout / dropout3 of layer l."""
import copy
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import avhubert_oracle as ao

from helpers import cosine, rel_err
from test_gpu_train_regularization import _check_grads, _encoder_step, _inputs, _loss, _Masks, _np_seed_dropping, _same

pytestmark = pytest.mark.gpu

REG = dict(dropout=0.2, activation_dropout=0.3, encoder_layerdrop=0.5)
TAIL_REG = dict(dropout_input=0.1, dropout=0.1, activation_dropout=0.1, encoder_layerdrop=0.5)


def _ref_encoder_postln(enc, x, pm, masks, skip, p_enc, p_act):
    """wav2vec2.py:859-902 / :993-1012 (post-LN) on the oracle's encoder modules with the step's masks and coins."""
    def drop(v, site, p):
        m = masks(site, tuple(v.shape), p)
        return v if m is None else v * m.to(v.dtype)

    if pm is not None:
        x = x.masked_fill(pm.unsqueeze(-1), 0.0)
    x = drop(enc.layer_norm(x + enc.pos_conv(x.transpose(1, 2)).transpose(1, 2)), 2, p_enc)
    for l, lyr in enumerate(enc.layers):
        if skip[l]:
            continue
        s = 16 + 4 * l
        a = lyr.self_attn(x.transpose(0, 1), pm).transpose(0, 1)
        x = lyr.self_attn_layer_norm(x + drop(a, s, p_enc))
        g = drop(F.gelu(lyr.fc1(x).float()).type_as(x), s + 1, p_act)
        x = lyr.final_layer_norm(x + drop(lyr.fc2(g), s + 2, p_enc))
    return x


def _ref_tail_postln(o, fused, pm, masks, skip, p_in, p_enc, p_act):
    """hubert.py:719-745 after the fusion: layer_norm -> post_extract_proj -> dropout_input -> post-LN encoder."""
    feats = o.layer_norm(fused)
    if o.post_extract_proj is not None:
        feats = o.post_extract_proj(feats)
    m = masks(1, tuple(feats.shape), p_in)
    if m is not None:
        feats = feats * m.to(feats.dtype)
    return _ref_encoder_postln(o.encoder, feats, pm, masks, skip, p_enc, p_act)


def _postln_pair(D, F_, H, L, seed, **reg):
    from multimodalvc_b200.sr_predictor import TransformerEncoder
    cfg = ao.OracleConfig(encoder_layers=L, encoder_embed_dim=D, encoder_ffn_embed_dim=F_, encoder_attention_heads=H,
                          layer_norm_first=False, conv_pos=128, conv_pos_groups=16)
    torch.manual_seed(seed)
    ref = ao._Encoder(cfg)
    ao.randomize_norm_stats(ref)
    with torch.no_grad():
        for m in ref.modules():
            if isinstance(m, torch.nn.Linear):
                m.weight.mul_(3.0)
    args = dict(dropout=0.0, attention_dropout=0.0, activation_dropout=0.0, encoder_layerdrop=0.0)
    args.update(reg)
    enc = TransformerEncoder(SimpleNamespace(encoder_embed_dim=D, encoder_ffn_embed_dim=F_, encoder_attention_heads=H,
                                             encoder_layers=L, conv_pos=128, conv_pos_groups=16, layer_norm_first=False,
                                             activation_fn="gelu", **args), trainable=True)
    enc.load_state_dict(ref.state_dict(), strict=True)
    return ref, enc


ENCODER_CASES = {
    "d128_plain": dict(D=128, F=256, H=2, L=2, B=2, T=37, lengths=[37, 20], reg={}, skip=[0, 0]),
    "d128_reg": dict(D=128, F=256, H=2, L=2, B=2, T=37, lengths=[37, 20], reg=REG, skip=[0, 1]),
    # the Speech_Rate_Predictor's encoder shape: D=256, F=1024, 4 heads
    "d256_plain": dict(D=256, F=1024, H=4, L=2, B=3, T=50, lengths=[50, 31, 44], reg={}, skip=[0, 0]),
    "d256_reg": dict(D=256, F=1024, H=4, L=2, B=3, T=50, lengths=[50, 31, 44], reg=REG, skip=[1, 0]),
}


@pytest.mark.parametrize("name", list(ENCODER_CASES))
def test_postln_encoder_step_matches_masked_autograd(name):
    case = ENCODER_CASES[name]
    L, reg = case["L"], case["reg"]
    ref, enc = _postln_pair(case["D"], case["F"], case["H"], L, seed=7, **reg)
    x, pm, w = _inputs(case["B"], case["T"], case["D"], case["lengths"], seed=8)
    enc = enc.cuda().train()
    np.random.seed(_np_seed_dropping(L, reg.get("encoder_layerdrop", 0.0), case["skip"]) if reg else 0)
    torch.manual_seed(11)
    xd = x.cuda().requires_grad_(True)
    y, _ = enc(xd, pm.cuda())
    seed, skip = enc._last_train_args
    assert skip == case["skip"] and (seed != 0) == bool(reg)
    _loss(y, w.cuda(), pm.cuda()).backward()
    r = copy.deepcopy(ref).double().train()
    xr = x.double().requires_grad_(True)
    y_ref = _ref_encoder_postln(r, xr, pm, _Masks(seed), skip, reg.get("dropout", 0.0), reg.get("activation_dropout", 0.0))
    _loss(y_ref, w.double(), pm).backward()
    assert rel_err(y.detach().cpu()[~pm], y_ref.detach()[~pm]) < 2e-3
    assert rel_err(xd.grad.cpu(), xr.grad) < 2e-3
    _check_grads(enc.named_parameters(), {n: p.grad for n, p in r.named_parameters()}, skip)


def _tiny_postln_model(fuse, fgm, reg, oracle_seed=1234):
    from multimodalvc_b200 import AVHubertConfig, AVHubertModel
    o = ao.build_oracle("tiny", seed=oracle_seed, modality_fuse=fuse, layer_norm_first=False).train()
    with torch.no_grad():
        for mod in o.encoder.modules():
            if isinstance(mod, torch.nn.Linear):
                mod.weight.mul_(3.0)
    cfg = AVHubertConfig.named("tiny", modality_fuse=fuse, feature_grad_mult=fgm, trainable=True, layer_norm_first=False,
                               attention_dropout=0.0, **reg)
    m = AVHubertModel(cfg)
    m.remove_pretraining_modules()
    m.load_state_dict(o.state_dict(), strict=False)
    return o, m.cuda().train()


@pytest.mark.parametrize("fuse", ["concat", "add"])
def test_postln_frozen_extractor_step_matches_masked_autograd_and_the_no_grad_training_forward(fuse):
    """Tail step (feature_grad_mult = 0) against the masked reference; then the no-grad training-mode forward with the
    same numpy / torch seeds gives the step's output: the two paths number their dropout sites alike in post-LN order."""
    o, m = _tiny_postln_model(fuse, 0.0, TAIL_REG)
    B, T, lengths = 3, 30, [30, 21, 26]
    src, pm = ao.synthetic_inputs(B, T, lengths=lengths, seed=13)
    w = torch.randn(B, T, 128, generator=torch.Generator().manual_seed(2)).masked_fill(pm.unsqueeze(-1), 0.0)
    dsrc = {k: v.cuda() for k, v in src.items()}
    nps = _np_seed_dropping(2, 0.5, [0, 1])
    np.random.seed(nps)
    torch.manual_seed(21)
    y, _ = m.extract_finetune(dsrc, pm.cuda())
    seed, skip = m._last_train_args
    assert skip == [0, 1]
    _loss(y, w.cuda(), pm.cuda()).backward()
    od = copy.deepcopy(o).double()
    with torch.no_grad():
        fv = od.feature_extractor_video(src["video"].double())
        fa = od.feature_extractor_audio(src["audio"].double())
        fused = (torch.cat([fa, fv], dim=1) if fuse == "concat" else fa + fv).transpose(1, 2)
    y_ref = _ref_tail_postln(od, fused, pm, _Masks(seed), skip, 0.1, 0.1, 0.1)
    _loss(y_ref, w.double(), pm).backward()
    assert rel_err(y.detach().cpu()[~pm], y_ref.detach()[~pm]) < 2e-3
    ref_grads = {n: p.grad for n, p in od.named_parameters()}
    for n, p in m.named_parameters():
        if n.startswith("feature_extractor"):
            assert p.grad is None, n
    _check_grads([(n, p) for n, p in m.named_parameters() if not n.startswith("feature_extractor")], ref_grads, skip)
    np.random.seed(nps)
    torch.manual_seed(21)
    with torch.no_grad():
        y_fwd, _ = m.extract_finetune(dsrc, pm.cuda())
    assert rel_err(y.detach().cpu()[~pm], y_fwd.cpu()[~pm]) < 2e-3


def test_postln_whole_model_step_matches_masked_autograd():
    """feature_grad_mult = 1: gradients outside the lip ResNet element-wise, the ResNet's with the statistical gates of
    the pre-LN whole-model test (its backward has kinks the fp32 forward can land on either side of)."""
    o32, m = _tiny_postln_model("concat", 1.0, TAIL_REG)
    B, T = 2, 16
    src32, pm = ao.synthetic_inputs(B, T, lengths=[16, 11], seed=19)
    w = torch.randn(B, T, 128, generator=torch.Generator().manual_seed(6))
    np.random.seed(_np_seed_dropping(2, 0.5, [1, 0]))
    torch.manual_seed(3)
    y, _ = m.extract_finetune({k: v.cuda() for k, v in src32.items()}, pm.cuda())
    seed, skip = m._last_train_args
    assert skip == [1, 0]
    _loss(y, w.cuda(), pm.cuda()).backward()
    o = copy.deepcopy(o32).double()
    src = {k: v.double() for k, v in src32.items()}
    fused = torch.cat([o.feature_extractor_audio(src["audio"]), o.feature_extractor_video(src["video"])], dim=1).transpose(1, 2)
    y_ref = _ref_tail_postln(o, fused, pm, _Masks(seed), skip, 0.1, 0.1, 0.1)
    _loss(y_ref, w.double(), pm).backward()
    assert rel_err(y.detach().cpu()[~pm], y_ref.detach()[~pm]) < 2e-3
    _check_grads(m.named_parameters(), {n: p.grad for n, p in o.named_parameters()}, skip,
                 stat_names=("feature_extractor_video.resnet",))


def test_postln_large_layer_bf16_step_and_device_weight_refresh():
    """D=1024, F=4096, 16 heads, one layer kept and one dropped, B=2, T=150: bf16 gradients against the masked fp32
    restatement (cosine >= 0.98); then in fp32 mode an SGD step on the library's gradients lowers the loss (the next step
    runs on weights refreshed in place on the device), that step's output is a fresh model's for the updated state
    dict, and so is the eval forward afterwards."""
    from multimodalvc_b200.sr_predictor import TransformerEncoder
    reg = dict(dropout=0.1, activation_dropout=0.1, encoder_layerdrop=0.5)
    ref, enc = _postln_pair(1024, 4096, 16, 2, seed=3, **reg)
    x, pm, w = _inputs(2, 150, 1024, [150, 97], seed=4)
    nps = _np_seed_dropping(2, 0.5, [0, 1])
    enc = enc.cuda().bfloat16().train()
    np.random.seed(nps)
    torch.manual_seed(8)
    xd = x.cuda().bfloat16().requires_grad_(True)
    y, _ = enc(xd, pm.cuda())
    seed, skip = enc._last_train_args
    assert skip == [0, 1]
    _loss(y.float(), w.cuda(), pm.cuda()).backward()
    r = copy.deepcopy(ref).train()
    xr = x.clone().requires_grad_(True)
    _loss(_ref_encoder_postln(r, xr, pm, _Masks(seed), skip, 0.1, 0.1), w, pm).backward()
    assert cosine(xd.grad.float().cpu(), xr.grad) > 0.98
    ref_grads = {n: p.grad for n, p in r.named_parameters()}
    for n, p in enc.named_parameters():
        if n.startswith("layers.1."):
            assert p.grad is None, n
        elif not n.endswith("k_proj.bias"):
            assert cosine(p.grad.float().cpu(), ref_grads[n]) > 0.98, (n, cosine(p.grad.float().cpu(), ref_grads[n]))
    enc = enc.float()
    opt = torch.optim.SGD(enc.parameters(), lr=0.5)

    def step(module):
        np.random.seed(nps)
        torch.manual_seed(8)
        yy, _ = module(x.cuda().requires_grad_(True), pm.cuda())
        return yy, _loss(yy, w.cuda(), pm.cuda())

    _, l0 = step(enc)
    l0.backward()
    opt.step()
    opt.zero_grad()
    y1, l1 = step(enc)
    assert l1.item() < l0.item()
    fresh = TransformerEncoder(enc.args, trainable=True)
    fresh.load_state_dict(enc.state_dict())
    fresh = fresh.cuda().train()
    y_fresh, _ = step(fresh)
    assert rel_err(y1.detach().cpu()[~pm], y_fresh.detach().cpu()[~pm]) < 1e-5
    with torch.no_grad():
        y_eval, _ = enc.eval()(x.cuda(), pm.cuda())
        y_eval_fresh, _ = fresh.eval()(x.cuda(), pm.cuda())
    assert rel_err(y_eval.cpu()[~pm], y_eval_fresh.cpu()[~pm]) < 1e-5


def test_postln_graph_replay_takes_the_seed_and_coins_of_each_step():
    from multimodalvc_b200 import _lib
    _, enc = _postln_pair(128, 256, 2, 2, seed=5, **REG)
    sd = copy.deepcopy(enc.state_dict())
    x, pm, w = _inputs(2, 40, 128, [40, 27], seed=9)
    keep, drop1 = _np_seed_dropping(2, 0.5, [0, 0]), _np_seed_dropping(2, 0.5, [0, 1])
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):                  # plan graphs are used on a non-default stream
        enc = enc.cuda().train()
        pmd, wd = pm.cuda(), w.cuda()
        first = _encoder_step(enc, x, pmd, wd, keep, 1)                 # direct
        second = _encoder_step(enc, x, pmd, wd, keep, 1)                # captured, then replayed
        g0 = _lib.load().avh_graph_launch_count()
        third = _encoder_step(enc, x, pmd, wd, keep, 1)                 # replayed
        assert _lib.load().avh_graph_launch_count() > g0
        _same(first, second)
        _same(first, third)
        other_seed = _encoder_step(enc, x, pmd, wd, keep, 2)            # replayed with another seed
        assert not torch.equal(other_seed[0], first[0])
        g1 = _lib.load().avh_graph_launch_count()
        replayed = _encoder_step(enc, x, pmd, wd, drop1, 1)             # layer 1 dropped, replayed
        assert _lib.load().avh_graph_launch_count() > g1
        assert enc._last_train_args[1] == [0, 1]
        assert all(replayed[2][n] is None for n in replayed[2] if n.startswith("layers.1."))
        for result, np_seed, torch_seed in ((other_seed, keep, 2), (replayed, drop1, 1)):
            _, fresh = _postln_pair(128, 256, 2, 2, seed=5, **REG)
            fresh.load_state_dict(sd)
            fresh = fresh.cuda().train()
            _same(result, _encoder_step(fresh, x, pmd, wd, np_seed, torch_seed))
