"""The pretraining step on the device: AVHubertModel.forward in .train() with gradients enabled (avhubert/hubert.py:591-674,
fairseq's av_hubert_pretraining task + hubert_criterion) — span masking, the two modality-dropout coins, features_pen,
the training step of the tail / whole model, final_proj and the cosine / dot logits, all differentiated on the device —
against torch.autograd in float64 on the oracle's modules, and the kernel-level backward of compute_logits."""
import copy
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import _GradMultiply, cosine, rel_err
from oracle import avhubert_oracle as ao
from oracle import pretrain_oracle as po

pytestmark = pytest.mark.gpu

NUM_CLASSES = [23, 17]
FINAL_DIM = 32
PEN_WEIGHT = 10.0          # hubert_criterion's loss_weights for features_pen in the shipped pretraining configs
MASK = dict(mask_prob_image=0.5, mask_length_image=5, mask_prob_audio=0.5, mask_length_audio=5)


def _cfg_kw(fuse, fgm, n_dicts, sim, selection, **kw):
    d = dict(modality_fuse=fuse, feature_grad_mult=fgm, trainable=True, dropout=0.0, attention_dropout=0.0,
             activation_dropout=0.0, encoder_layerdrop=0.0, dropout_input=0.0, final_dim=FINAL_DIM,
             untie_final_proj=n_dicts > 1, sim_type=sim, selection_type=selection, logit_temp=0.1,
             modality_dropout=0.5, audio_dropout=0.5, **MASK)
    d.update(kw)
    return d


def _head(n_dicts, D, seed):
    g = torch.Generator().manual_seed(seed)
    rows = FINAL_DIM * (n_dicts if n_dicts > 1 else 1)
    w = torch.randn(rows, D, generator=g) * 0.1
    b = torch.randn(rows, generator=g) * 0.1
    embs = torch.rand(sum(NUM_CLASSES[:n_dicts]), FINAL_DIM, generator=g)
    return w, b, embs


def _device_model(o32, head, size, dtype, **kw):
    import types
    from multimodalvc_b200 import AVHubertConfig, AVHubertModel
    n_dicts = 2 if kw.get("untie_final_proj") else 1      # one tied dictionary or two untied ones
    cfg = AVHubertConfig.named(size, **kw)
    m = AVHubertModel(cfg, types.SimpleNamespace(sample_rate=25), [list(range(n)) for n in NUM_CLASSES[:n_dicts]])
    sd = dict(o32.state_dict())
    sd["final_proj.weight"], sd["final_proj.bias"], sd["label_embs_concat"] = head
    sd["mask_emb"] = torch.rand(m.mask_emb.shape, generator=torch.Generator().manual_seed(3))
    missing = m.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and not missing.missing_keys, missing
    return m.to(device="cuda", dtype=dtype).train()


def _po_head(m, n_dicts):
    c = m.cfg
    return po.Head(m.mask_emb.detach().float().cpu(), m.final_proj.weight.detach().float().cpu(),
                   m.final_proj.bias.detach().float().cpu(), m.label_embs_concat.detach().float().cpu(), NUM_CLASSES[:n_dicts],
                   **MASK, sim_type=c.sim_type, selection_type=c.selection_type, untie_final_proj=n_dicts > 1)


def _draws(head, src, pm):
    """The host side of one step in the reference's order on the CPU: span masks (video, then audio), the two modality
    coins.  Returns (masked video, masked audio, mask_indices, (modality coin, audio coin))."""
    from multimodalvc_b200 import masking
    v, mv = po.apply_input_mask(head, src["video"].clone(), pm, masking.compute_mask_indices)
    a, ma = po.apply_input_mask(head, src["audio"].clone(), pm, masking.compute_mask_indices)
    return v, a, mv | ma, (np.random.random(), np.random.random())


def _decision(coins, modality_dropout=0.5, audio_dropout=0.5):
    return 0 if coins[0] >= modality_dropout else (1 if coins[1] < audio_dropout else 2)


def _seed(s):
    np.random.seed(s)
    torch.manual_seed(s)


def _np_seed_dropping(head, src, pm, want, start=0):
    """A seed whose two modality coins, drawn after the step's span masks, drop `want` (0 none, 1 audio, 2 video)."""
    for s in range(start, start + 1000):
        _seed(s)
        if _decision(_draws(head, src, pm)[3]) == want:
            return s
    raise AssertionError("no seed found")


def _ref_step(o, head, v, a, pm, mi, targets, fgm, fuse, drop, n_dicts, sim, temp=0.1):
    """hubert.py:591-674 in training mode on the oracle's modules (float64), the criterion's loss: sum of the
    cross-entropies over masked and unmasked frames of every dictionary + PEN_WEIGHT * features_pen."""
    w, b, embs = head

    def features(extractor, x):
        if fgm > 0:
            f = extractor(x)
            return _GradMultiply.apply(f, fgm) if fgm != 1.0 else f
        with torch.no_grad():
            return extractor(x)

    fv = features(o.feature_extractor_video, v)
    fa = features(o.feature_extractor_audio, a)
    if drop == 1:
        fa = 0 * fa
    elif drop == 2:
        fv = 0 * fv
    feats = torch.cat([fa, fv], dim=1) if fuse == "concat" else fa + fv
    pen = feats.pow(2).mean()
    x = o.layer_norm(feats.transpose(1, 2))
    if o.post_extract_proj is not None:
        x = o.post_extract_proj(x)
    x = o.encoder(x, pm)
    proj = x @ w.t() + b
    projs = proj.chunk(n_dicts, dim=-1) if n_dicts > 1 else [proj] * len(NUM_CLASSES[:n_dicts])
    logits = [_logits(p, e, sim, temp).view(-1, n)
              for p, e, n in zip(projs, embs.split(NUM_CLASSES[:n_dicts], 0), NUM_CLASSES[:n_dicts])]
    sel_m, sel_u = (mi & ~pm).view(-1), (~mi & ~pm).view(-1)
    lm = [lg[sel_m] for lg in logits]
    lu = [lg[sel_u] for lg in logits]
    return lm, lu, pen, _loss(lm, lu, pen, targets, sel_m, sel_u)


def _logits(f, e, sim, temp):
    """pretrain_oracle.compute_logits in the inputs' dtype (the oracle's computes in fp32)."""
    lead = f.shape[:-1]
    f = f.reshape(-1, f.size(-1))
    if sim == "dot":
        return (f @ e.t()).view(*lead, -1) / temp
    den = f.pow(2).sum(-1).sqrt()[:, None] * e.pow(2).sum(-1).sqrt()[None, :]
    return ((f @ e.t()) / den.clamp(min=1e-6)).view(*lead, -1) / temp


def _loss(lm, lu, pen, targets, sel_m, sel_u):
    loss = 0
    for i, t in enumerate(targets):
        t = t.reshape(-1).to(lm[i].device)
        loss = loss + F.cross_entropy(lm[i].double(), t[sel_m.to(t.device)], reduction="sum")
        loss = loss + F.cross_entropy(lu[i].double(), t[sel_u.to(t.device)], reduction="sum")
    return loss + PEN_WEIGHT * pen.double()


def _targets(B, T, n_dicts, seed=5):
    g = torch.Generator().manual_seed(seed)
    return [torch.randint(0, n, (B, T), generator=g) for n in NUM_CLASSES[:n_dicts]]


CASES = [
    # fuse, feature_grad_mult, modality dropped (0 none, 1 audio, 2 video), dictionaries (2 = untied), sim, selection
    ("concat", 1.0, 0, 1, "cosine", "same_other_seq"),
    ("concat", 1.0, 2, 2, "dot", "same_seq"),
    ("concat", 0.1, 1, 1, "cosine", "same_seq"),
    ("add", 1.0, 1, 2, "cosine", "same_other_seq"),
    ("add", 0.1, 2, 1, "dot", "same_other_seq"),
    ("add", 0.0, 0, 2, "dot", "same_seq"),
    ("concat", 0.0, 2, 1, "cosine", "same_other_seq"),
    ("concat", 0.0, 1, 2, "cosine", "same_seq"),
]


@pytest.mark.parametrize("fuse,fgm,drop,n_dicts,sim,selection", CASES)
def test_pretraining_step_matches_autograd(fuse, fgm, drop, n_dicts, sim, selection):
    """fp32 mode, tiny model, ragged batch: logits, features_pen and every gradient against float64 autograd on the oracle
    (the gates of test_full_finetune_step_matches_autograd: PReLU slopes 1, so the trunk is judged element-wise and the
    stem — behind the max-pool — statistically); the dropped extractor's gradients are zeros (not None), its BatchNorm
    running statistics move as the oracle's; numpy's generator ends where the reference's does."""
    B, T, lengths = 2, 16, [16, 11]
    o32 = ao.build_oracle("tiny", seed=1234, modality_fuse=fuse).train()
    for mod in o32.modules():
        if isinstance(mod, torch.nn.PReLU):
            mod.weight.data.fill_(1.0)
    head32 = _head(n_dicts, 128, seed=9)
    m = _device_model(o32, head32, "tiny", torch.float32, **_cfg_kw(fuse, fgm, n_dicts, sim, selection))
    src, pm = ao.synthetic_inputs(B, T, lengths=lengths, seed=19)
    targets = _targets(B, T, n_dicts)
    ph = _po_head(m, n_dicts)
    seed = _np_seed_dropping(ph, src, pm, drop)
    # reference: the same draws on the CPU, then the coins of the encoder's LayerDrop (drawn whatever the probability)
    _seed(seed)
    v, a, mi, coins = _draws(ph, src, pm)
    assert _decision(coins) == drop
    for _ in range(m.cfg.encoder_layers):
        np.random.random()
    want_next = np.random.random()
    o = copy.deepcopy(o32).double()
    head = tuple(t.double().requires_grad_(True) for t in head32)
    lm_r, lu_r, pen_r, loss_r = _ref_step(o, head, v.double(), a.double(), pm, mi, targets, fgm, fuse, drop, n_dicts, sim)
    loss_r.backward()
    # device
    _seed(seed)
    dsrc = {k: t.cuda() for k, t in src.items()}
    res = m(dsrc, target_list=[t.cuda() for t in targets], padding_mask=pm.cuda(), mask=True)
    assert np.random.random() == want_next          # span masks + 2 modality coins + LayerDrop coins, nothing else
    for i in range(n_dicts):
        assert res["logit_m_list"][i].grad_fn is not None and res["logit_u_list"][i].grad_fn is not None
        assert rel_err(res["logit_m_list"][i].detach().cpu(), lm_r[i].detach()) < 2e-3
        assert rel_err(res["logit_u_list"][i].detach().cpu(), lu_r[i].detach()) < 2e-3
    pen = res["features_pen"]
    assert abs(pen.item() - pen_r.item()) <= 1e-5 * pen_r.item()
    assert (pen.grad_fn is not None) == (fgm > 0)
    sel_m = (mi & ~pm).view(-1).cuda()
    sel_u = (~mi & ~pm).view(-1).cuda()
    _loss(res["logit_m_list"], res["logit_u_list"], pen, [t.cuda() for t in targets], sel_m, sel_u).backward()
    # gradients
    ref = {n: p.grad for n, p in o.named_parameters()}
    ref["final_proj.weight"], ref["final_proj.bias"], ref["label_embs_concat"] = (t.grad for t in head)
    dropped = {1: "feature_extractor_audio.", 2: "feature_extractor_video."}.get(drop)
    bad = {}
    for n, p in m.named_parameters():
        if n == "mask_emb" or ref.get(n) is None:
            assert p.grad is None or not p.grad.any(), n
            continue
        assert p.grad is not None, n
        g = p.grad.cpu().double()
        if dropped is not None and n.startswith(dropped) and fgm > 0:
            assert not g.any() and not ref[n].any(), n          # 0 * features: zero gradients, not None
            continue
        r = ref[n]
        if n.endswith("k_proj.bias"):       # exactly 0 in exact arithmetic: judged on q_proj.bias' scale
            err = (g - r).abs().max().item() / ref[n.replace("k_proj", "q_proj")].abs().max().item()
        elif "frontend3D" in n:             # behind the max-pool: statistical gate
            l2 = ((g - r).norm() / r.norm()).item()
            if l2 > 3e-2 or cosine(g, r) < 0.9995:
                bad[n] = f"rel-L2 {l2:.2e} cosine {cosine(g, r):.6f}"
            continue
        else:
            err = rel_err(g, r)
        if err > 2e-3:
            bad[n] = f"max-abs {err:.2e}"
    assert not bad, "\n".join(f"{k}: {v}" for k, v in bad.items())
    if fgm <= 0:
        assert all(p.grad is None for n, p in m.named_parameters() if n.startswith("feature_extractor"))
    # BatchNorm running statistics (the video extractor runs even when its features are dropped)
    for name in ("frontend3D.1", "trunk.layer2.0.bn1", "trunk.layer4.1.bn2"):
        bn_o = o.feature_extractor_video.resnet.get_submodule(name)
        bn_m = m.feature_extractor_video.resnet.get_submodule(name)
        assert (bn_m.running_mean.cpu() - bn_o.running_mean).abs().max().item() < 1e-4, name
        assert (bn_m.running_var.cpu() - bn_o.running_var).abs().max().item() < 1e-4, name


def _step(m, src, pm, targets, seed):
    """One pretraining step from `seed` with the criterion's loss (mean cross-entropies here)."""
    _seed(seed)
    res = m(src, target_list=targets, padding_mask=pm, mask=True)
    loss = res["features_pen"] * PEN_WEIGHT
    for i in range(len(targets)):
        loss = loss + F.cross_entropy(res["logit_m_list"][i], res["target_m_list"][i]) + \
            F.cross_entropy(res["logit_u_list"][i], res["target_u_list"][i])
    return res, loss


def test_pretraining_step_bf16_large_and_sgd():
    """bf16 mode at the Large layer shape (2 x 24 frames): gradient directions against autograd on the oracle (fp32, on
    the GPU), and three SGD steps on the same batch lower the loss."""
    B, T, lengths = 2, 24, [24, 17]
    o32 = ao.build_oracle("large", seed=1234)
    head32 = _head(1, 1024, seed=4)
    kw = _cfg_kw("concat", 1.0, 1, "cosine", "same_other_seq", final_dim=FINAL_DIM, modality_dropout=0.0)
    m = _device_model(o32.train(), head32, "large", torch.bfloat16, **kw)
    src, pm = ao.synthetic_inputs(B, T, lengths=lengths, seed=29)
    targets = _targets(B, T, 1)
    ph = _po_head(m, 1)
    _seed(3)
    v, a, mi, _ = _draws(ph, src, pm)
    o = copy.deepcopy(o32).cuda().train()
    head = tuple(t.cuda().requires_grad_(True) for t in head32)
    _, _, _, loss_r = _ref_step(o, head, v.cuda(), a.cuda(), pm.cuda(), mi.cuda(), targets, 1.0, "concat", 0, 1, "cosine")
    loss_r.backward()
    ref = {n: p.grad.double().cpu() for n, p in o.named_parameters() if p.grad is not None}
    ref["final_proj.weight"], ref["final_proj.bias"], ref["label_embs_concat"] = (t.grad.double().cpu() for t in head)
    del o
    dsrc = {k: t.cuda().bfloat16() for k, t in src.items()}
    _seed(3)
    res = m(dsrc, target_list=[t.cuda() for t in targets], padding_mask=pm.cuda(), mask=True)
    sel_m = (mi & ~pm).view(-1).cuda()
    sel_u = (~mi & ~pm).view(-1).cuda()
    _loss(res["logit_m_list"], res["logit_u_list"], res["features_pen"], [t.cuda() for t in targets], sel_m, sel_u).backward()
    low, worst = {}, {}
    for n, p in m.named_parameters():
        if n == "mask_emb" or ref.get(n) is None or n.endswith("k_proj.bias"):
            continue
        c = cosine(p.grad.float().cpu().double(), ref[n])
        gate = 0.90 if (".relu" in n or n.endswith("frontend3D.2.weight")) else (0.93 if "resnet" in n else 0.97)
        kind = "resnet" if "resnet" in n else "other"
        worst[kind] = min(worst.get(kind, 1.0), c)
        if c < gate:
            low[n] = c
    print(f"bf16 Large pretraining step: worst cosine {worst}")
    assert not low, low
    opt = torch.optim.SGD(m.parameters(), lr=0.01)
    tg = [t.cuda() for t in targets]
    losses = []
    for _ in range(3):
        opt.zero_grad()
        _, loss = _step(m, dsrc, pm.cuda(), tg, seed=3)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print(f"bf16 Large pretraining SGD losses {losses}")
    assert losses[2] < losses[1] < losses[0], losses


def test_graph_replay_and_train_to_eval():
    """Consecutive steps on a side stream (the plan's CUDA graphs replayed) with the drop decisions none -> video ->
    audio -> none and different seeds: outputs and gradients bit-identical to the same steps on freshly built models;
    then the eval-mode forward after training equals that of a fresh model loaded from the state dict."""
    B, T, lengths = 2, 16, [16, 12]
    o32 = ao.build_oracle("tiny", seed=1234).train()
    head32 = _head(2, 128, seed=9)
    kw = _cfg_kw("concat", 1.0, 2, "cosine", "same_other_seq", capture_stages=True)
    src, pm = ao.synthetic_inputs(B, T, lengths=lengths, seed=31)
    targets = _targets(B, T, 2)
    m = _device_model(o32, head32, "tiny", torch.bfloat16, **kw)
    ph = _po_head(m, 2)
    seeds = [_np_seed_dropping(ph, src, pm, d) for d in (0, 2, 1)]
    seeds.append(_np_seed_dropping(ph, src, pm, 0, start=seeds[0] + 1))
    dsrc = {k: t.cuda().bfloat16() for k, t in src.items()}
    dpm = pm.cuda()
    tg = [t.cuda() for t in targets]

    def run(model, seed):
        model.zero_grad(set_to_none=True)
        res, loss = _step(model, dsrc, dpm, tg, seed)
        loss.backward()
        torch.cuda.synchronize()
        out = [lg.detach().clone() for lg in res["logit_m_list"] + res["logit_u_list"]] + [res["features_pen"].detach()]
        grads = {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}
        return out, grads

    side = torch.cuda.Stream()
    got = []
    with torch.cuda.stream(side):
        for s in seeds:
            got.append(run(m, s))
    torch.cuda.synchronize()
    for s, (out, grads) in zip(seeds, got):
        fresh = _device_model(o32, head32, "tiny", torch.bfloat16, **kw)
        with torch.cuda.stream(side):
            want_out, want_grads = run(fresh, s)
        for x, y in zip(out, want_out):
            assert torch.equal(x, y), s
        assert grads.keys() == want_grads.keys()
        for n in grads:
            assert torch.equal(grads[n], want_grads[n]), (s, n)
        del fresh
    # train -> eval through the device-side refresh: an SGD update on the last step's gradients, and the BatchNorm running
    # statistics the four steps moved
    with torch.no_grad():
        for p in m.parameters():
            if p.grad is not None:
                p -= 0.01 * p.grad
    m.eval()
    fresh = _device_model(o32, head32, "tiny", torch.bfloat16, **kw)
    fresh.load_state_dict(m.state_dict())
    fresh.eval()
    _seed(77)
    with torch.no_grad():
        r1 = m(dsrc, target_list=tg, padding_mask=dpm, mask=True)
    _seed(77)
    with torch.no_grad():
        r2 = fresh(dsrc, target_list=tg, padding_mask=dpm, mask=True)
    for x, y in zip(r1["logit_m_list"] + r1["logit_u_list"], r2["logit_m_list"] + r2["logit_u_list"]):
        assert torch.equal(x, y)
    assert torch.equal(r1["features_pen"], r2["features_pen"])


@pytest.mark.parametrize("M,V,K,sim,bias,f_dt", [
    (1, 23, 32, "cosine", False, torch.float32),
    (1, 5, 7, "dot", True, torch.float32),
    (150, 504, 256, "cosine", False, torch.float32),
    (97, 70, 129, "dot", True, torch.float32),
    (64, 65, 63, "cosine", True, torch.bfloat16),
    (200, 17, 1024, "dot", False, torch.bfloat16),
    (1200, 40, 256, "cosine", True, torch.float32),       # dE split over m (partial sums added in order)
    (40, 1200, 64, "cosine", False, torch.float32),       # dF split over v
    (600, 300, 96, "dot", False, torch.bfloat16),
])
def test_compute_logits_backward_kernel(M, V, K, sim, bias, f_dt):
    """avh_compute_logits_backward against float64 autograd: M = 1, V and K off the 64 tiles, zero-norm rows (the clamp),
    bf16 features, with and without a bias, contractions split over their long axis; repeat calls are bit-identical."""
    from multimodalvc_b200 import _lib
    g = torch.Generator().manual_seed(M * 7 + V)
    f = torch.randn(M, K, generator=g).to(f_dt).float()
    e = torch.randn(V, K, generator=g)
    b = torch.randn(V, generator=g) if bias else None
    if M > 2:
        f[1] = 0                                         # zero-norm feature row: the clamped denominator is a constant
        e[2] = 0
    dl = torch.randn(M, V, generator=g)
    temp = 0.1 if sim == "cosine" else 1.0
    # reference: float64 with norms whose gradient at 0 is 0 (the reference's sqrt(sum x^2) gives 0 * inf there)
    fr, er = f.double().requires_grad_(True), e.double().requires_grad_(True)
    br = b.double().requires_grad_(True) if bias else None
    s = fr @ er.t() + (br if bias else 0)
    if sim == "cosine":
        den = torch.linalg.vector_norm(fr, dim=1)[:, None] * torch.linalg.vector_norm(er, dim=1)[None, :]
        s = s / den.clamp(min=1e-6)
    out_r = s / temp
    out_r.backward(dl.double())
    fd = f.to(f_dt).cuda()
    ed, dld = e.cuda(), dl.cuda()
    bd = b.cuda() if bias else None
    lg = torch.empty(M, V, device="cuda")
    lib = _lib.load()
    vp = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    dt = _lib.AVH_BF16 if f_dt == torch.bfloat16 else _lib.AVH_F32
    simc = 1 if sim == "cosine" else 0
    _lib.check(lib.avh_compute_logits(vp(fd), dt, K, vp(ed), _lib.AVH_F32, K, vp(bd), M, V, K, simc, temp, vp(lg), V, st))
    assert rel_err(lg.cpu(), out_r.detach()) < 1e-5
    outs = []
    for _ in range(2):
        df = torch.empty(M, K, device="cuda")
        de = torch.empty(V, K, device="cuda")
        db = torch.empty(V, device="cuda") if bias else None
        _lib.check(lib.avh_compute_logits_backward(vp(fd), dt, K, vp(ed), _lib.AVH_F32, K, M, V, K, simc, temp, vp(lg), vp(dld), V,
                                                   vp(df), K, vp(de), K, vp(db), st))
        outs.append((df, de, db))
    torch.cuda.synchronize()
    df, de, db = outs[0]
    assert torch.equal(df, outs[1][0]) and torch.equal(de, outs[1][1])
    # a zero-norm row's gradient is the dot term over the clamped denominator (1e6 times the others'): judged on its own
    zf = torch.zeros(M, dtype=torch.bool)
    ze = torch.zeros(V, dtype=torch.bool)
    if M > 2:
        zf[1], ze[2] = True, True
    for got, want, z in ((df.cpu(), fr.grad, zf), (de.cpu(), er.grad, ze)):
        assert rel_err(got[~z], want[~z]) < 2e-5, rel_err(got[~z], want[~z])
        if z.any():
            assert rel_err(got[z], want[z]) < 2e-5, rel_err(got[z], want[z])
    if bias:
        assert torch.equal(db, outs[1][2])
        assert rel_err(db.cpu(), br.grad) < 2e-5
    with pytest.raises(RuntimeError, match="logits"):       # the cosine backward reads the forward's logits
        _lib.check(lib.avh_compute_logits_backward(vp(fd), dt, K, vp(ed), _lib.AVH_F32, K, M, V, K, 1, temp, None, vp(dld), V,
                                                   vp(df), K, None, K, None, st))


def test_pretraining_step_errors():
    """What the training-mode pretraining forward leaves out raises as documented."""
    B, T = 2, 12
    o32 = ao.build_oracle("tiny", seed=1234).train()
    head32 = _head(1, 128, seed=9)
    src, pm = ao.synthetic_inputs(B, T, lengths=[12, 9], seed=5)
    dsrc = {k: t.cuda() for k, t in src.items()}
    tg = [t.cuda() for t in _targets(B, T, 1)]
    kw = _cfg_kw("concat", 1.0, 1, "cosine", "same_other_seq")
    with pytest.raises(NotImplementedError):                                       # attention dropout
        _device_model(o32, head32, "tiny", torch.float32, **dict(kw, attention_dropout=0.1))(dsrc, tg, pm.cuda())
    with pytest.raises(NotImplementedError):                                       # feature masking
        _device_model(o32, head32, "tiny", torch.float32, **dict(kw, masking_type="feature"))(dsrc, tg, pm.cuda())
    m = _device_model(o32, head32, "tiny", torch.float32, **kw)
    with pytest.raises(NotImplementedError):
        m(dsrc, tg, pm.cuda(), features_only=True)
    with pytest.raises(NotImplementedError):
        m(dsrc, tg, pm.cuda(), output_layer=1)
    with pytest.raises(NotImplementedError):                                       # under no_grad
        with torch.no_grad():
            m(dsrc, tg, pm.cuda())
    with pytest.raises(ValueError):                                                # single modality
        m({"audio": None, "video": dsrc["video"]}, tg, pm.cuda())
    with pytest.raises(NotImplementedError):                                       # not trainable
        _device_model(o32, head32, "tiny", torch.float32, **dict(kw, trainable=False))(dsrc, tg, pm.cuda())
    # the C entry points check their state
    from multimodalvc_b200 import _lib
    lib = _lib.load()
    assert lib.avh_set_modality_drop(m._ensure_handle(), 3) != 0
    assert lib.avh_set_features_pen_grad(m._ensure_handle(), None, None) != 0      # no pretraining step before it
