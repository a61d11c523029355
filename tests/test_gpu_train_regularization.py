"""Dropout, activation dropout and LayerDrop in the device training step (avh_set_train_args; TransformerEncoder and
AVHubertModel.extract_finetune in .train() with gradients enabled).

The library's masks are its own Philox stream (not torch's), so the reference here is the oracle's modules restated as
the pre-LN layer of wav2vec2.py with the step's masks injected at the reference's dropout sites and its LayerDrop coins
applied, differentiated by torch.autograd.  Every mask is rebuilt exactly with avh_dropout (same seed, same site id) on
a tensor of ones: site 1 dropout_input (hubert.py:729), 2 after the positional conv block (wav2vec2.py:879), 16+4l /
17+4l / 18+4l dropout1 / activation dropout / dropout3 of layer l (wav2vec2.py:980,987,990)."""
import copy
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import avhubert_oracle as ao

from helpers import cosine, rel_err

pytestmark = pytest.mark.gpu


def _loss(y, w, pm):
    valid = y if pm is None else y.masked_fill(pm.unsqueeze(-1), 0.0)
    return (valid * w).sum() / w.numel() + valid.pow(2).mean()


def _np_seed_dropping(n_layers, layerdrop, want):
    """A numpy seed whose first n_layers draws give the LayerDrop decisions `want` (1 = dropped)."""
    for s in range(10000):
        coins = np.random.RandomState(s).random_sample(n_layers)
        if [0 if c > layerdrop else 1 for c in coins] == list(want):
            return s
    raise AssertionError("no seed found")


class _Masks:
    """mask(site, rows, C, p) = the library's dropout mask of a site, [rows, C] fp32 on the CPU (None when p = 0)."""

    def __init__(self, seed):
        from multimodalvc_b200 import _lib
        self.lib, self.lib_mod, self.seed = _lib.load(), _lib, seed

    def __call__(self, site, shape, p):
        if p == 0.0:
            return None
        n = 1
        for d in shape:
            n *= d
        m = torch.ones(n, device="cuda", dtype=torch.float32)
        st = torch.cuda.current_stream().cuda_stream
        self.lib_mod.check(self.lib.avh_dropout(ctypes.c_void_p(m.data_ptr()), self.lib_mod.AVH_F32, n, p, self.seed, site,
                                                ctypes.c_void_p(st)))
        return m.cpu().view(shape)


def _ref_encoder(enc, x, pm, masks, skip, p_enc, p_act):
    """wav2vec2.py:859-902 / :974-992 (pre-LN) on the oracle's encoder modules with the step's masks and coins."""
    def drop(v, site, p):
        m = masks(site, tuple(v.shape), p)
        return v if m is None else v * m.to(v.dtype)

    if pm is not None:
        x = x.masked_fill(pm.unsqueeze(-1), 0.0)
    x = drop(x + enc.pos_conv(x.transpose(1, 2)).transpose(1, 2), 2, p_enc)
    for l, lyr in enumerate(enc.layers):
        if skip[l]:
            continue
        s = 16 + 4 * l
        a = lyr.self_attn(lyr.self_attn_layer_norm(x).transpose(0, 1), pm).transpose(0, 1)
        x = x + drop(a, s, p_enc)
        g = drop(F.gelu(lyr.fc1(lyr.final_layer_norm(x)).float()).type_as(x), s + 1, p_act)
        x = x + drop(lyr.fc2(g), s + 2, p_enc)
    return enc.layer_norm(x)


def _ref_tail(o, fused, pm, masks, skip, p_in, p_enc, p_act):
    """hubert.py:719-745 after the fusion: layer_norm -> post_extract_proj -> dropout_input -> encoder."""
    feats = o.layer_norm(fused)
    if o.post_extract_proj is not None:
        feats = o.post_extract_proj(feats)
    m = masks(1, tuple(feats.shape), p_in)
    if m is not None:
        feats = feats * m.to(feats.dtype)
    return _ref_encoder(o.encoder, feats, pm, masks, skip, p_enc, p_act)


def _encoder_pair(D, F_, H, L, seed, **reg):
    from multimodalvc_b200.sr_predictor import TransformerEncoder
    cfg = ao.OracleConfig(encoder_layers=L, encoder_embed_dim=D, encoder_ffn_embed_dim=F_, encoder_attention_heads=H,
                          layer_norm_first=True, conv_pos=128, conv_pos_groups=16)
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
                                             encoder_layers=L, conv_pos=128, conv_pos_groups=16, layer_norm_first=True,
                                             activation_fn="gelu", **args), trainable=True)
    enc.load_state_dict(ref.state_dict(), strict=True)
    return ref, enc


def _inputs(B, T, D, lengths, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, D, generator=g)
    pm = None if lengths is None else torch.arange(T)[None, :] >= torch.tensor(lengths)[:, None]
    w = torch.randn(B, T, D, generator=g)
    if pm is not None:
        w = w.masked_fill(pm.unsqueeze(-1), 0.0)
    return x, pm, w


def _check_grads(named, ref_grads, skip, strict_names=None, stat_names=()):
    """Every parameter gradient against the reference (2e-3 of the tensor's maximum; k_proj.bias on q_proj.bias' scale;
    `stat_names`: cosine >= 0.9995 and relative L2 <= 3e-2); parameters of dropped layers have no gradient."""
    bad = {}
    for n, p in named:
        layer = n.split("layers.")[1].split(".")[0] if "layers." in n else None
        if layer is not None and skip[int(layer)]:
            assert p.grad is None, n
            continue
        if n == "mask_emb" or n not in ref_grads or ref_grads[n] is None:
            continue
        assert p.grad is not None, n
        a, r = p.grad.cpu().double(), ref_grads[n].double()
        if n.endswith("k_proj.bias"):
            err = (a - r).abs().max().item() / ref_grads[n.replace("k_proj", "q_proj")].abs().max().item()
            if err > 2e-3:
                bad[n] = err
        elif any(s in n for s in stat_names):
            l2 = ((a - r).norm() / r.norm()).item()
            if l2 > 3e-2 or cosine(a, r) < 0.9995:
                bad[n] = (l2, cosine(a, r))
        elif rel_err(a, r) > 2e-3:
            bad[n] = rel_err(a, r)
    assert not bad, bad


@pytest.mark.parametrize("case", [
    # the Speech_Rate_Predictor's encoder: D=256, F=1024, 4 heads, activation_dropout 0.1, LayerDrop 0.1 (layer 0 dropped)
    dict(D=256, F=1024, H=4, L=2, B=3, T=50, lengths=[50, 31, 44], reg=dict(activation_dropout=0.1, encoder_layerdrop=0.1),
         skip=[1, 0]),
    dict(D=128, F=256, H=2, L=2, B=2, T=37, lengths=[37, 20], reg=dict(dropout=0.2, activation_dropout=0.3), skip=[0, 0]),
])
def test_encoder_step_with_dropout_and_layerdrop_matches_masked_autograd(case):
    L, reg = case["L"], case["reg"]
    ref, enc = _encoder_pair(case["D"], case["F"], case["H"], L, seed=7, **reg)
    x, pm, w = _inputs(case["B"], case["T"], case["D"], case["lengths"], seed=8)
    enc = enc.cuda().train()
    np.random.seed(_np_seed_dropping(L, reg.get("encoder_layerdrop", 0.0), case["skip"]))
    torch.manual_seed(11)
    xd = x.cuda().requires_grad_(True)
    y, _ = enc(xd, pm.cuda())
    seed, skip = enc._last_train_args
    assert skip == case["skip"] and seed != 0
    _loss(y, w.cuda(), pm.cuda()).backward()
    r = copy.deepcopy(ref).double().train()
    xr = x.double().requires_grad_(True)
    y_ref = _ref_encoder(r, xr, pm, _Masks(seed), skip, reg.get("dropout", 0.0), reg.get("activation_dropout", 0.0))
    _loss(y_ref, w.double(), pm).backward()
    assert rel_err(y.detach().cpu()[~pm], y_ref.detach()[~pm]) < 2e-3
    assert rel_err(xd.grad.cpu(), xr.grad) < 2e-3
    _check_grads(enc.named_parameters(), {n: p.grad for n, p in r.named_parameters()}, skip)


def _tiny_model(fuse, fgm, reg, oracle_seed=1234):
    from multimodalvc_b200 import AVHubertConfig, AVHubertModel
    o = ao.build_oracle("tiny", seed=oracle_seed, modality_fuse=fuse).train()
    with torch.no_grad():
        for mod in o.encoder.modules():
            if isinstance(mod, torch.nn.Linear):
                mod.weight.mul_(3.0)
    cfg = AVHubertConfig.named("tiny", modality_fuse=fuse, feature_grad_mult=fgm, trainable=True, attention_dropout=0.0, **reg)
    m = AVHubertModel(cfg)
    m.remove_pretraining_modules()
    m.load_state_dict(o.state_dict(), strict=False)
    return o, m.cuda().train()


TAIL_REG = dict(dropout_input=0.1, dropout=0.1, activation_dropout=0.1, encoder_layerdrop=0.5)


def test_frozen_extractor_step_matches_masked_autograd_and_the_no_grad_training_forward():
    """Tail step (feature_grad_mult = 0, concat fusion) against the masked reference; then the no-grad training-mode
    forward (avh_forward_train) with the same numpy / torch seeds draws the same coins and seed and gives the same
    output: the two paths number their dropout sites alike."""
    o, m = _tiny_model("concat", 0.0, TAIL_REG)
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
        fused = torch.cat([fa, fv], dim=1).transpose(1, 2)
    y_ref = _ref_tail(od, fused, pm, _Masks(seed), skip, 0.1, 0.1, 0.1)
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


def test_whole_model_step_matches_masked_autograd():
    """feature_grad_mult = 1: gradients outside the lip ResNet element-wise, the ResNet's with the statistical gates of
    test_full_finetune_step_matches_autograd (its backward has kinks the fp32 forward can land on either side of)."""
    o32, m = _tiny_model("concat", 1.0, TAIL_REG)
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
    y_ref = _ref_tail(o, fused, pm, _Masks(seed), skip, 0.1, 0.1, 0.1)
    _loss(y_ref, w.double(), pm).backward()
    assert rel_err(y.detach().cpu()[~pm], y_ref.detach()[~pm]) < 2e-3
    _check_grads(m.named_parameters(), {n: p.grad for n, p in o.named_parameters()}, skip,
                 stat_names=("feature_extractor_video.resnet",))


def test_training_steps_draw_only_the_layerdrop_coins():
    """Per step the numpy stream advances by exactly encoder_layers draws (the reference's coins), in the
    frozen-extractor step (whose stage pre-pass draws nothing) and in the whole-model step alike."""
    _, m0 = _tiny_model("concat", 0.0, TAIL_REG)
    _, m1 = _tiny_model("concat", 1.0, TAIL_REG)
    src, pm = ao.synthetic_inputs(2, 12, lengths=[12, 9], seed=3)
    dsrc = {k: v.cuda() for k, v in src.items()}
    np.random.seed(77)
    m0.extract_finetune(dsrc, pm.cuda())[0].sum().backward()
    m1.extract_finetune(dsrc, pm.cuda())[0].sum().backward()
    after = np.random.random()
    np.random.seed(77)
    np.random.random(2 * 2)
    assert np.random.random() == after


def _encoder_step(enc, x, pm, w, np_seed, torch_seed):
    enc.zero_grad()
    np.random.seed(np_seed)
    torch.manual_seed(torch_seed)
    xd = x.cuda().requires_grad_(True)
    y, _ = enc(xd, pm)
    _loss(y, w, pm).backward()
    torch.cuda.synchronize()
    return y.detach().clone(), xd.grad.clone(), {n: (p.grad.clone() if p.grad is not None else None)
                                                 for n, p in enc.named_parameters()}


def _same(a, b):
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for n in a[2]:
        assert (a[2][n] is None) == (b[2][n] is None), n
        assert a[2][n] is None or torch.equal(a[2][n], b[2][n]), n


def test_graph_replay_takes_the_seed_and_coins_of_each_step():
    from multimodalvc_b200 import _lib
    reg = dict(dropout=0.2, activation_dropout=0.3, encoder_layerdrop=0.5)
    _, enc = _encoder_pair(128, 256, 2, 2, seed=5, **reg)
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
        other_seed = _encoder_step(enc, x, pmd, wd, keep, 2)
        assert not torch.equal(other_seed[0], first[0])
        g1 = _lib.load().avh_graph_launch_count()
        replayed = _encoder_step(enc, x, pmd, wd, drop1, 1)             # layer 1 dropped, replayed
        assert _lib.load().avh_graph_launch_count() > g1
        assert enc._last_train_args[1] == [0, 1]
        assert all(replayed[2][n] is None for n in replayed[2] if n.startswith("layers.1."))
        _, fresh = _encoder_pair(128, 256, 2, 2, seed=5, **reg)
        fresh.load_state_dict(sd)
        fresh = fresh.cuda().train()
        direct = _encoder_step(fresh, x, pmd, wd, drop1, 1)
        _same(replayed, direct)


def test_zero_regularization_runs_the_plain_step():
    """avh_set_train_args with every probability 0 and no coins selects the plan of a step without the call: the same
    launches, the same graph segments, bit-identical gradients."""
    from multimodalvc_b200 import _lib, _train
    _, enc = _encoder_pair(128, 256, 2, 2, seed=5)
    x, pm, w = _inputs(2, 40, 128, [40, 27], seed=9)
    side = torch.cuda.Stream()
    lib = _lib.load()

    def counted_step():
        l0, g0 = lib.avh_launch_count(), lib.avh_graph_launch_count()
        out = _encoder_step(enc, x, pmd, wd, 0, 0)
        return out, lib.avh_launch_count() - l0, lib.avh_graph_launch_count() - g0

    with torch.cuda.stream(side):
        enc = enc.cuda().train()
        pmd, wd = pm.cuda(), w.cuda()
        with_call = [counted_step() for _ in range(3)]
        orig = _train.StepRegularization.set_on
        _train.StepRegularization.set_on = lambda self, handle: None
        try:
            without = [counted_step() for _ in range(3)]
        finally:
            _train.StepRegularization.set_on = orig
    assert with_call[2][1] == without[2][1] and with_call[2][2] == without[2][2] and with_call[2][2] > 0
    _same(with_call[0][0], without[2][0])


def test_large_layer_bf16_with_dropout_and_layerdrop():
    """D=1024, F=4096, 16 heads: one layer kept and one dropped, B=2, T=150, bf16: every gradient against the masked fp32
    restatement (cosine >= 0.98); an SGD step on the library's gradients, seed and coins held fixed, lowers the loss."""
    reg = dict(dropout=0.1, activation_dropout=0.1, encoder_layerdrop=0.5)
    ref, enc = _encoder_pair(1024, 4096, 16, 2, seed=3, **reg)
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
    _loss(_ref_encoder(r, xr, pm, _Masks(seed), skip, 0.1, 0.1), w, pm).backward()
    assert cosine(xd.grad.float().cpu(), xr.grad) > 0.98
    ref_grads = {n: p.grad for n, p in r.named_parameters()}
    for n, p in enc.named_parameters():
        if n.startswith("layers.1."):
            assert p.grad is None, n
        elif not n.endswith("k_proj.bias"):
            assert cosine(p.grad.float().cpu(), ref_grads[n]) > 0.98, (n, cosine(p.grad.float().cpu(), ref_grads[n]))
    enc = enc.float()
    opt = torch.optim.SGD(enc.parameters(), lr=0.5)

    def step_loss():
        np.random.seed(nps)
        torch.manual_seed(8)
        yy, _ = enc(x.cuda().requires_grad_(True), pm.cuda())
        return _loss(yy, w.cuda(), pm.cuda())

    l0 = step_loss()
    l0.backward()
    opt.step()
    opt.zero_grad()
    assert step_loss().item() < l0.item()
